"""Benchmark of the generator hot path (BASELINE.json configs[1]):

  BaseGen default chain -- GMM intensities + affine/nonlinear deformation + gamma + bias field + resolution
  degradation (blur, downsample, noise, re-upsample, normalise) + the always-on T1 target warp --
  batch 8 x 160^3 per step on each GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  `value` = samples/s with all inputs resident in HBM (host-side random
draws and table planning INCLUDED, overlapped with the GPU through the asynchronous stream); `e2e` = the same
through the public API with host label/image buffers copied in and the generated volumes copied out every
step; `roofline` = the dominant kernel (warp+gamma+bias) against the measured HBM peak; `cpu_baseline` = the
oracle port of the reference's PyTorch-CPU generator on this box's host cores.

`--dump-outputs DIR` writes what the device-resident arm's last timed step handed its caller (rank 0): every tensor of
the batch's samples and targets, stacked over the batch, as DIR/<name>.npy in float32 (see `dump_outputs`).  The
inputs and the random streams depend on the arguments only, so two builds run with the same arguments can be
compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np   # noqa: E402
import torch         # noqa: E402

SIZE = 160
BATCH = 8
METRIC = "synthetic 160^3 samples/sec (BaseGen default chain, batch 8)"
UNIT = "samples/s"


class quiet_gc:
    """Timed regions run with Python's cyclic collector off (what `timeit` does): a generation-2 collection over the
    heap of an imported torch takes 5-200 ms and lands deterministically inside a 20-step region (measured: ONE step
    of 206 ms among 0.3 ms steps; profiles/README.md, 'host-side stalls').  The current heap is frozen first so that
    later collections stay cheap."""

    def __enter__(self):
        import gc
        gc.collect()
        gc.freeze()
        gc.disable()
        return self

    def __exit__(self, *exc):
        import gc
        gc.enable()
        return False


def make_inputs(n_subjects):
    """Subjects of the bench: label map = the 160^3 crop of round(files/gca.mgz) SURVEY.md 8d names (committed as
    tests/golden/atlas_gca_L160_u8.npz -- the reference tree does not exist on the GPU box), shifted by a few voxels per
    subject so that the subjects are distinct volumes; T1 = the atlas intensities themselves.  Label maps are integer
    valued (uint8 on the wire and in HBM); T1 is int16, the dtype T1w NIfTI / FreeSurfer volumes are stored in -- it
    crosses PCIe as 2 bytes per voxel and is widened on the device (bfm_ingest_volume)."""
    from tests import _inputs as ti
    shp = (SIZE, SIZE, SIZE)
    fixture = os.path.join(ROOT, "tests", "golden", "atlas_gca_L160_u8.npz")
    atlas = np.load(fixture)["L160"] if os.path.exists(fixture) and SIZE <= 160 else None
    if atlas is not None and SIZE < 160:
        o = (160 - SIZE) // 2
        atlas = atlas[o:o + SIZE, o:o + SIZE, o:o + SIZE]
    subs = []
    for s in range(n_subjects):
        if atlas is None:
            subs.append(dict(Gen=ti.brain_like_labels(shp, seed=7 + s),
                             T1=np.round(ti.smooth_image(shp, 0.1 * s)).astype(np.int16)))
            continue
        lab = np.roll(atlas, shift=(s + 1) // 2 * (1 if s % 2 else -1), axis=s % 3)
        subs.append(dict(Gen=lab.astype(np.float32), T1=lab.astype(np.int16)))
    return subs


def bench_cfg():
    from tests import _inputs as ti
    cfg = ti.default_cfg((SIZE,) * 3)
    for k in vars(cfg.task):
        setattr(cfg.task, k, False)          # "tasks off": input (+ BFlog written) + the unconditional T1 target
    return cfg


def ncu_traffic(kernel_prefix):
    """dram__bytes_read + dram__bytes_write (bytes per launch) of the newest committed ncu full capture."""
    import csv
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_full_v*_summary.csv")),
                   key=lambda p: [int(t) for t in __import__("re").findall(r"\d+", os.path.basename(p))])
    for path in reversed(files):
        try:
            rows = list(csv.reader(open(path)))
            hdr, units = rows[0], rows[1]
            ir, iw = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
            scale = {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}
            vals = [float(r[ir]) * scale[units[ir]] + float(r[iw]) * scale[units[iw]] for r in rows[2:]
                    if r[0].replace("void ", "").startswith(kernel_prefix)]
            if vals:
                return float(np.mean(vals)), os.path.basename(path)
        except Exception:
            continue
    return None, None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons (B200_PROFILING.md recipe), sampled every 20 ms from BEFORE the warm-up
    (nvidia-smi needs ~100 ms to come up) until the end of the run.  Every line is time-stamped on arrival;
    `summary(t0, t1)` reports the samples that fell inside the timed region [t0, t1] and, beside them, all samples
    taken under load (warm-up through the end-to-end arm) -- the device-resident timed region of the default
    run lasts only ~30 ms."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        if os.environ.get("BFM_CLOCK_MS") == "0":       # development switch: no sampler at all
            return
        # in-process NVML: 5 ms period, so that a timed region of ~14 ms (20 steps) holds 2-3 samples
        self.period = float(os.environ.get("BFM_CLOCK_MS", "5")) * 1e-3
        self._stop = False
        # in-process NVML (three queries per sample) when pynvml is importable; an `nvidia-smi -lms` child otherwise.
        # The child re-queries a dozen fields per line through the driver and was measured to cost the two-stream
        # device-resident arm ~5-8 % at a 20 ms period.
        try:
            if os.environ.get("BFM_CLOCK_SMI") == "1":
                raise RuntimeError("nvidia-smi forced")
            import pynvml
            pynvml.nvmlInit()
            self.nvml, self.handle = pynvml, pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
            self.nvml.nvmlDeviceGetClockInfo(self.handle, self.nvml.NVML_CLOCK_SM)
            self.proc = "nvml"
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", os.environ.get("BFM_CLOCK_MS", "20")],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if self.index < len(ids) and ids[self.index].isdigit():
                return int(ids[self.index])
        return self.index

    def _poll(self):
        n = self.nvml
        bits = [("hw_slowdown", getattr(n, "nvmlClocksEventReasonHwSlowdown", 0x8)),
                ("hw_thermal_slowdown", getattr(n, "nvmlClocksEventReasonHwThermalSlowdown", 0x40)),
                ("sw_thermal_slowdown", getattr(n, "nvmlClocksEventReasonSwThermalSlowdown", 0x20)),
                ("sw_power_cap", getattr(n, "nvmlClocksEventReasonSwPowerCap", 0x4))]
        get_reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(n, "nvmlDeviceGetCurrentClocksThrottleReasons")
        try:
            mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        except Exception:
            mx = 0
        while not self._stop:
            try:
                sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                r = int(get_reasons(self.handle))
                row = [str(sm), str(mx)] + ["Active" if r & b else "Not Active" for _, b in bits]
                self.rows.append((time.perf_counter(), row))
            except Exception:
                pass
            time.sleep(self.period)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def wait_first(self, timeout=3.0):
        t_end = time.perf_counter() + timeout
        while self.proc is not None and not self.rows and time.perf_counter() < t_end:
            time.sleep(0.01)

    def stop(self):
        if self.proc is None:
            return
        if self.proc == "nvml":
            self._stop = True
            return
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()

    def _stats(self, rows):
        rows = [r for _, r in rows if len(r) >= 6]
        sm = [float(r[0]) for r in rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if r[1].replace(".", "").isdigit()]
        reasons = sorted({self.NAMES[i] for r in rows for i in range(4) if r[2 + i].startswith("Active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}

    def summary(self, t0, t1, load0, load1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        timed = self._stats([r for r in self.rows if t0 <= r[0] <= t1])
        load = self._stats([r for r in self.rows if load0 <= r[0] <= load1])
        out = dict(timed if timed["samples"] else load)
        out["sampler"] = "nvml (in-process)" if self.proc == "nvml" else "nvidia-smi -lms"
        out["window"] = "timed region" if timed["samples"] else "whole run under load (timed region < sampling interval)"
        out["timed_region_samples"] = timed["samples"]
        out["under_load"] = load
        return out


# ------------------------------------------------------------------------------------------------ reference arm
def oracle_generator(subs, threads):
    from oracle import gen_oracle as go
    torch.set_num_threads(threads)
    gens = [go.GeneratorOracle(bench_cfg(), {k: np.asarray(v, dtype=np.float32) for k, v in s.items()}) for s in subs]
    return gens


def time_oracle(gens, n_samples, seed=0):
    from oracle import gen_oracle as go
    go.seed_all(seed)
    t0 = time.perf_counter()
    for i in range(n_samples):
        gens[i % len(gens)].sample()
    return time.perf_counter() - t0


def run_reference(args, rank, world):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    gens = oracle_generator(make_inputs(2), threads)
    t1 = time_oracle(gens, 1, seed=123)            # page-in / first-touch
    t1 = time_oracle(gens, 1, seed=124)
    budget = 150.0
    per_step = int(max(1, min(BATCH, budget / max(t1, 1e-3) / (args.steps + args.warmup))))
    for _ in range(args.warmup):
        time_oracle(gens, per_step)
    t0 = time.perf_counter()
    for k in range(args.steps):
        time_oracle(gens, per_step, seed=k)
    dt = time.perf_counter() - t0
    val = args.steps * per_step / dt
    sample = "%d of the %d samples of a step (160^3 each), %d steps" % (per_step, BATCH, args.steps)
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def config_dict():
    return {"workload": "configs[1]: BaseGen default chain batch 8x160^3 (GMM + affine/nonlinear deform + gamma + "
                        "bias + blur/downsample/noise/upsample/normalise + T1 target warp), tasks off, label maps = 160^3 "
                        "crop of round(files/gca.mgz) (SURVEY 8d; committed fixture tests/golden/atlas_gca_L160_u8.npz), T1 = "
                        "the atlas intensities (int16), reference parameter ranges (default.yaml + train/brain_id.yaml)",
            "batch": BATCH, "size": [SIZE] * 3, "source": [SIZE] * 3,
            "l2": "working set per step (8 samples x ~100 MB of intermediates) exceeds the 126 MB L2; "
                  "no explicit flush",
            "rng": "scalars: library planner (bfm_plan_batch), Philox4x32-10 stream seeded from numpy's global "
                   "generator, reference draw order and distributions; small random grids and volume-sized normal "
                   "fields: in-kernel Philox4x32-10"}


def bind_to_gpu_numa_node(index):
    """One process per GPU: run on the CPUs of the GPU's NUMA node, so that the pinned host buffers of the end-to-end
    arm (first touch) and the planner live next to the GPU's PCIe root.  Returns the node, or None if unknown."""
    try:
        bus = torch.cuda.get_device_properties(index).pci_bus_id
        dom = torch.cuda.get_device_properties(index).pci_domain_id
        dev = torch.cuda.get_device_properties(index).pci_device_id
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (dom, bus, dev)
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------ our arm
def build_dataset(subs, device, planner="auto"):
    from brainfm_b200 import io as bio
    from brainfm_b200.Generator import BaseGen
    root = tempfile.mkdtemp(prefix="bfm_bench_")
    names = []
    for s, v in enumerate(subs):
        stem = os.path.join(root, "HCP.sub%02d." % s)
        bio.register_volume(stem + "T1w.nii", v["T1"])
        bio.register_volume(stem + "generation_labels.nii", v["Gen"])
        names.append(stem + "T1w.nii")
    with open(os.path.join(root, "train.txt"), "w") as f:
        f.write("\n".join(names) + "\n")
    cfg = bench_cfg()
    cfg.split_root = root
    ds = BaseGen(cfg, device, planner=planner)
    ds.write_bflog = True
    return ds


DUMP_BYTES = 64_000_000


def batch_outputs(items):
    """The tensors a caller receives from one batch, stacked over its items: those of the samples (`input`,
    `bias_field_log`, ...) and those of the targets (`target_T1`, ...)."""
    out = {}
    for _, _, _, target, sample in items:
        for smp in sample if isinstance(sample, list) else [sample]:
            for k, v in smp.items():
                if torch.is_tensor(v):
                    out.setdefault(k, []).append(v)
        for k, v in target.items():
            if torch.is_tensor(v):
                out.setdefault("target_" + k, []).append(v)
    return {k: torch.stack(v) for k, v in out.items()}


def dump_outputs(arrays, path):
    """Writes every array as <path>/<name>.npy in float32, DUMP_BYTES in all.  An array larger than its equal share is
    flattened and sampled: the same seeded, sorted set of flat indices for every array of that size, so that the
    samples of, say, `input` and `bias_field_log` are the same voxels."""
    os.makedirs(path, exist_ok=True)
    share = (DUMP_BYTES // max(1, len(arrays)) - 1024) // 4          # float32 values per array (1 KB for the header)
    picks = {}
    for name, t in sorted(arrays.items()):
        a = t.detach().to(torch.float32).cpu().numpy()
        if a.size > share:
            if a.size not in picks:
                picks[a.size] = np.sort(np.random.default_rng(0).choice(a.size, share, replace=False))
            a = a.reshape(-1)[picks[a.size]]
        np.save(os.path.join(path, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="device-resident arm only (profiling runs)")
    ap.add_argument("--planner", default="auto", choices=["auto", "python", "native"])
    ap.add_argument("--lanes", type=int, default=2, help="batches in flight in the device-resident arm")
    ap.add_argument("--no-extras", action="store_true", help="skip the configs[2..4] records")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step of the device-resident arm as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs the CUDA path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch.distributed as dist
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    # one process per GPU: run (and first-touch the pinned buffers) on the GPU's NUMA node unless BFM_NUMA_BIND=0
    numa = bind_to_gpu_numa_node(local) if world > 1 and os.environ.get("BFM_NUMA_BIND", "1") != "0" else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner on stdout when the communicator comes up: send fd 1 to stderr meanwhile, so
        # that stdout carries nothing but the one JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=device)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    from brainfm_b200 import _lib
    n_subjects = 2 * BATCH          # the end-to-end arm alternates between two sets of subjects
    subs = make_inputs(n_subjects)
    ds = build_dataset(subs, device, args.planner)
    from brainfm_b200 import parallel as par
    # the path shards by sample: every rank generates its own stream of batches (disjoint random streams),
    # there is no data-path collective; only the timing below is reduced (max over ranks)
    np.random.seed(par.rank_seed(1000, rank))
    torch.manual_seed(par.rank_seed(1000, rank))
    idxs = list(range(BATCH))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident arm ----------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        ds.generate_batch(idxs)
    barrier()
    if rank == 0:
        sampler.wait_first()
    for _ in range(args.warmup):           # nvidia-smi came up while rank 0 idled: back under load before timing
        ds.generate_batch(idxs)
    barrier()
    load_t0 = time.perf_counter()
    # `value`: the public device-resident API (brainfm_b200.pipeline.DevicePipeline): two batches in flight, each on
    # its own stream with its own scratch; every step plans, launches and hands over one batch of 8
    from brainfm_b200.pipeline import DevicePipeline
    dpipe = DevicePipeline(ds, depth=args.lanes)
    tickets = []
    # untimed: the pipeline's own warm-up, in the same submit / wait rhythm as the timed loop (a one-off host stall of
    # 1.5-200 ms was measured at the pipeline's 8th submit whatever the path -- see profiles/README.md)
    for _ in range(max(2 * args.lanes, int(os.environ.get("BFM_PIPE_WARMUP", "16")))):
        tickets.append(dpipe.submit(idxs))
        if len(tickets) > args.lanes:
            tickets.pop(0).wait()
    for t in tickets:
        t.wait()
    tickets = []
    t = None          # the loop variable would keep the last warm-up batch's outputs alive through the timed loop: one
    #                   more live set than the warm-up ever had => three cudaMallocs (1.3-200 ms) at the third timed step
    barrier()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    gcq = quiet_gc().__enter__()
    barrier()
    e0.record()
    wait0 = ds.arena.wait_s
    t0 = time.perf_counter()
    tickets = []
    trace = [] if os.environ.get("BFM_BENCH_TRACE") == "1" else None
    if trace is not None:
        ds._trace = []
    for k in range(args.steps):
        if trace is not None:
            ts = time.perf_counter()
        tickets.append(dpipe.submit(idxs))
        if len(tickets) > args.lanes:
            tickets.pop(0).wait()                # the consumer's stream takes the batch (stream wait, no host sync)
        if trace is not None:
            trace.append(round(1e3 * (time.perf_counter() - ts), 3))
            tr = getattr(ds, '_trace', None)
            if rank == 0 and k < 6:
                ms_ = torch.cuda.memory_stats()
                print("step %d: segments %d, cudaMalloc retries %d, reserved %.2f GB, active %.2f GB, host %.3f ms" %
                      (k, ms_.get("segment.all.current", -1), ms_.get("num_alloc_retries", -1),
                       ms_.get("reserved_bytes.all.current", 0) / 1e9, ms_.get("active_bytes.all.current", 0) / 1e9,
                       trace[-1]), file=sys.stderr, flush=True)
            if tr and trace[-1] > 1.0 and rank == 0:
                print("slow step %d: %s (whole step %.3f ms)" % (k, [(a, round(1e3 * (b - tr[0][1]), 3)) for a, b in tr],
                                                                 trace[-1]), file=sys.stderr, flush=True)
    for t in tickets:
        t.wait()
    e1.record()
    barrier()
    t1 = time.perf_counter()
    gcq.__exit__()
    if args.dump_outputs and rank == 0:
        dump_outputs(batch_outputs(tickets[-1].items), args.dump_outputs)
    host_s = t1 - t0
    if trace is not None and rank == 0:
        print("per-step host ms: %s" % trace, file=sys.stderr, flush=True)
    host_wait_s = ds.arena.wait_s - wait0        # of which: waiting for a free plan-arena slot, i.e. for the GPU
    launches = _lib.launch_count() - l0
    dev_ms = e0.elapsed_time(e1)
    # stage breakdown + the dominant kernel's launch duration: a second pass of the same K steps on ONE stream with
    # CUDA events around every stage (events between the stages of two interleaved streams would time the other
    # stream's kernels too)
    timers = {}
    for k in range(args.steps):
        ds.generate_batch(idxs, timers=timers)
    barrier()
    el = torch.tensor([dev_ms], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(el, op=dist.ReduceOp.MAX)
    total_ms = float(el.item())
    value = world * args.steps * BATCH / (total_ms * 1e-3)

    stage_ms = {k: float(np.mean([a.elapsed_time(b) for a, b in v])) for k, v in timers.items()}

    # ---------------- algorithmic bytes of the dominant kernel (warp + gamma + bias + T1 target) ----------------
    # per sample: gather-read of the GMM image and of the T1 volume over the bbox crop (2 * 4*Nc) + write I_bf,
    # BFlog and the raw warped T1 (3 * 4*N)
    N = SIZE ** 3
    np.random.seed(par.rank_seed(1000, rank))
    torch.manual_seed(par.rank_seed(1000, rank))
    items = ds.generate_batch(idxs)
    nc = []
    ns = []
    if ds._native is not None:
        for bb, new in ds._native.last_shapes():
            nc.append((bb[3] - bb[0]) * (bb[4] - bb[1]) * (bb[5] - bb[2]))
            ns.append(int(np.prod(new)))
    else:
        for j in ds._last_jobs:
            bb = j["plan"].bbox_host()
            nc.append((bb[3] - bb[0]) * (bb[4] - bb[1]) * (bb[5] - bb[2]))
            ns.append(int(np.prod(j["p"]["new_size"])))
    nc_mean, ns_mean = float(np.mean(nc)), float(np.mean(ns))
    peak, peak_src = peaks()
    warp_bytes = BATCH * (8 * nc_mean + 12 * N)
    warp_ms = stage_ms.get("warp", float("nan"))
    achieved = warp_bytes / (warp_ms * 1e-3) / 1e9
    # SURVEY 8d: 4Nc + 16N + 12Ns for the synthetic chain, + (4Nc + 4N) for the T1 target warp
    chain_bytes = 4 * nc_mean + 16 * N + 12 * ns_mean + (4 * nc_mean + 4 * N)
    chain_gbs = chain_bytes * value / world / 1e9

    traffic, traffic_src = ncu_traffic("k_gen_warp_pk")
    if args.quick:
        sampler.stop()
        if rank == 0:
            print(json.dumps({"quick": True, "value": value, "host_wall_ms_per_step": 1e3 * host_s / args.steps,
                              "host_busy_ms_per_step": 1e3 * (host_s - host_wait_s) / args.steps,
                              "stage_ms_per_step": stage_ms}), flush=True)
        return
    # ---------------- end-to-end arm: host buffers in, host buffers out ----------------
    # Every step uploads the label map (uint8) and the T1 volume (int16, its stored dtype) of its 8 subjects from pinned host
    # memory and downloads the 8 generated volumes into pinned host memory, through the public pipelined API
    # (brainfm_b200.pipeline.HostPipeline): the upload of step k+1 and the download of step k-1 overlap the
    # generation of step k, so consecutive steps alternate between two sets of 8 subjects.
    from brainfm_b200.pipeline import HostPipeline
    # host side of a step: one pinned (8, 160^3) uint8 label batch and one pinned (8, 160^3) int16 T1 batch (what a
    # collating loader hands over); each is ONE host->device DMA, the results come back as one (8, 1, 160^3) DMA
    sets = [list(range(0, BATCH)), list(range(BATCH, 2 * BATCH))]
    host_lab = [torch.from_numpy(np.stack([subs[s]["Gen"].astype(np.uint8) for s in st])).pin_memory() for st in sets]
    host_t1 = [torch.from_numpy(np.stack([subs[s]["T1"] for s in st])).pin_memory() for st in sets]       # int16
    uploads = [[([ds.names[0][s][:-7] + "generation_labels.nii" for s in st], "gen", host_lab[q]),
                ([ds.names[0][s] for s in st], "f32", host_t1[q])] for q, st in enumerate(sets)]
    h2d = host_lab[0].numel() * host_lab[0].element_size() + host_t1[0].numel() * host_t1[0].element_size()
    d2h = BATCH * SIZE ** 3 * 4
    pipe = HostPipeline(ds, depth=3)

    def e2e_run(n):
        tickets = []
        for k in range(n):
            tickets.append(pipe.submit(sets[k % 2], uploads[k % 2]))
            if len(tickets) > 2:
                tickets.pop(0).wait()
        for t in tickets:
            t.wait()

    # warm-up of the end-to-end arm (untimed): the first passes on a fresh box run at a fraction of the steady PCIe
    # rate (first touch of ~0.8 GB of pinned memory, link and clock ramp-up), so keep going until two consecutive
    # blocks of 8 steps agree within 5 % (at most ~4 s)
    e2e_run(4)
    prev, t_begin, series = None, time.perf_counter(), []
    while time.perf_counter() - t_begin < 4.0:
        torch.cuda.synchronize()
        w0 = time.perf_counter()
        e2e_run(8)
        torch.cuda.synchronize()
        cur = (time.perf_counter() - w0) / 8
        series.append(round(1e3 * cur, 3))
        if prev is not None and abs(cur - prev) <= 0.05 * prev and len(series) >= 3:
            break
        prev = cur
    if rank == 0:
        print("e2e warm-up ms/step per block of 8: %s" % series, file=sys.stderr, flush=True)
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with quiet_gc():
        f0.record()
        e2e_run(args.steps)
        torch.cuda.synchronize()
        f1.record()
    barrier()
    el2 = torch.tensor([f0.elapsed_time(f1)], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(el2, op=dist.ReduceOp.MAX)
    e2e_value = world * args.steps * BATCH / (float(el2.item()) * 1e-3)
    load_t1 = time.perf_counter()
    clocks = None
    if rank == 0:
        sampler.stop()
        clocks = sampler.summary(t0, t1, load_t0, load_t1)

    # ---------------- the other BASELINE.json configurations, on the record (extra keys, not bench values) ----------------
    # (before the CPU baseline: after ~4 s of 16 busy host threads the host-paced ShapeID solver loop was measured at
    # twice its time)
    extras = {}
    if not args.no_extras:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        gcx = quiet_gc().__enter__()
        try:
            if world == 1:
                import config_bench as cb
                r = cb.interpol_cfg(256)                      # configs[2]
                r["frac_of_peak"] = r["algorithmic_GBps"] / peak
                extras["interpol256"] = r
                r = cb.shapeid_cfg(192)                       # configs[3]
                r["frac_of_peak"] = r["algorithmic_GBps"] / peak
                extras["shapeid192"] = r
                extras["brainid_stream"] = cb.brainid_cfg()   # configs[4]a
            else:
                import slab_bench as sb                       # configs[4]b: one 512^3 volume in x-slabs over the ranks
                extras["slab512"] = sb.run(512, 6, rank, world, local)
                extras["slab512"].pop("profile", None)
        except Exception as e:                                # never lose the bench line over an extra
            extras["error"] = repr(e)[:300]
        gcx.__exit__()

    # ---------------- CPU baseline (oracle port), rank 0 at N=1 only ----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        gens = oracle_generator(subs[:2], threads)
        time_oracle(gens, 1, seed=5)
        n = 12
        dt = time_oracle(gens, n, seed=6)
        cpu = {"value": n / dt, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": "%d samples of 160^3 (same label maps, same parameter ranges), torch %d threads" % (n, threads)}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_dict(),
                "roofline": {"bound": "hbm", "kernel": "k_gen_warp_pk (paired gather of synth + T1, gamma, bias; batch 8)",
                             "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": warp_bytes, "ms_per_launch": warp_ms},
                "chain": {"algorithmic_bytes_per_sample": chain_bytes, "achieved_gbs": chain_gbs,
                          "frac_of_peak": chain_gbs / peak, "nc_over_n": nc_mean / N, "ns_over_n": ns_mean / N,
                          "stage_ms_per_step": stage_ms, "host_wall_ms_per_step": 1e3 * host_s / args.steps,
                          "host_busy_ms_per_step": 1e3 * (host_s - host_wait_s) / args.steps},
                "cpu_baseline": cpu,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
                "gpu_launches": int(launches), "clocks": clocks, "configs": extras}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
