"""Device-resident throughput of generate_batch without per-stage events (development tool, not a bench value)."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import bench
from brainfm_b200 import _lib

STEPS = int(os.environ.get("STEPS", "30"))


def main():
    dev = torch.device("cuda", 0)
    nstreams = int(os.environ.get("STREAMS", "1"))
    subs = bench.make_inputs(bench.BATCH)
    dss = [bench.build_dataset(subs, dev) for _ in range(nstreams)]
    streams = [torch.cuda.Stream() for _ in range(nstreams)]
    np.random.seed(1000)
    torch.manual_seed(1000)
    idxs = list(range(bench.BATCH))
    for k in range(6 * nstreams):
        with torch.cuda.stream(streams[k % nstreams]):
            dss[k % nstreams].generate_batch(idxs)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for st in streams:
        st.wait_event(e0)
    for k in range(STEPS):
        with torch.cuda.stream(streams[k % nstreams]):
            dss[k % nstreams].generate_batch(idxs)
    for st in streams:
        ev = torch.cuda.Event()
        ev.record(st)
        torch.cuda.current_stream().wait_event(ev)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / STEPS
    print(json.dumps({"ms_per_step": round(ms, 4), "samples_per_s": round(bench.BATCH / ms * 1e3, 1),
                      "streams": nstreams, "lib": os.path.basename(_lib.LIB_PATH)}))


if __name__ == "__main__":
    main()
