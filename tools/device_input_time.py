#!/usr/bin/env python
"""Device-resident input against the other two ways in, on bench.py's config 2 workload (same
generator, same seed): 4.6 Mbp synthetic reference, 20 000 reads, full-read mapping.

  map_device    the raw samples in a CUDA tensor (copied there once), smb_map_reads_device
  map_uploaded  smb_reads_upload once, then smb_map_uploaded (bench.py's `value`)
  map_reads     pinned host buffers, smb_map_reads: the samples cross PCIe in every call (`e2e`)

One process, one context.  Each path gets one warm-up call, then --rounds rounds call the three
in turn, so that drift of the card or the host touches all of them alike.  A call's time is the
library's device stopwatch (smb_timer_start/stop, as bench.py) and the host wall clock around the
call (every call returns synchronised); the rate is the call's consumed samples (stats `samples`)
over the device time.  Medians over the rounds.  The rows of all three paths must be identical,
byte for byte; the script fails otherwise.  Prints one JSON line (and writes it to --out), with
the card's name, power limit and SM clocks read in the same run."""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info(device):
    if not shutil.which("nvidia-smi"):
        return {"nvidia_smi": "unavailable"}
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", str(device)],
                         capture_output=True, text=True).stdout.strip()
    return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--reads", type=int, default=None, help="default: config 2's 20 000")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    import torch

    import bench
    from sigmap_b200.mapper import Mapper, full_read_params

    w = bench.resolve_workload(argparse.Namespace(
        workload="c2", shard="reads", ref_bp=None, contigs=None, reads=args.reads, mode=None, noise=1.0,
        seed=20251017, steps=3, cpu_sample_reads=1, ref_step_reads=1), 1)  # bench.py's default --seed
    H, model, ref, pos, val, reads = bench.build_workload(w, 0)
    assert w.mode == "full"
    params = full_read_params()
    dev = torch.device("cuda", args.device)
    m = Mapper(args.device)
    m.set_index(pos, val)
    m.set_contigs(ref.lengths)
    pinned = torch.empty(len(reads.raw), dtype=torch.int16, pin_memory=True)
    pinned.numpy()[:] = reads.raw
    reads.raw = pinned.numpy()
    raw_dev = pinned.to(dev)
    start = reads.read_off[:-1].copy()
    length = np.diff(reads.read_off).astype(np.uint32)
    torch.cuda.synchronize(dev)

    paths = {
        "map_device": lambda: m.map_device(raw_dev, start, length, reads.digitisation, reads.range, reads.offset,
                                           params),
        "map_uploaded": lambda: m.map_uploaded(params),
        "map_reads": lambda: m.map_reads(reads, params),
    }

    def call(name):
        if name == "map_uploaded":
            m.upload_reads(reads)  # untimed; map_device leaves no uploaded read set behind
        m.stats_reset()
        m.timer_start()
        t0 = time.perf_counter()
        rows = paths[name]()
        wall = time.perf_counter() - t0
        ms = m.timer_stop()
        st = m.stats()
        return rows, ms, wall * 1000.0, st

    info_before = gpu_info(args.device)
    rows = {}
    for name in paths:
        rows[name] = call(name)[0]
    times = {name: {"ms": [], "wall_ms": [], "samples": None, "h2d_bytes": None} for name in paths}
    for _ in range(args.rounds):
        for name in paths:
            r, ms, wall, st = call(name)
            rows[name] = r
            t = times[name]
            t["ms"].append(ms)
            t["wall_ms"].append(wall)
            t["samples"], t["h2d_bytes"] = int(st["samples"]), int(st["h2d_bytes"])
    info_after = gpu_info(args.device)

    as_bytes = {name: [bytes(x) for x in r] for name, r in rows.items()}
    identical = as_bytes["map_device"] == as_bytes["map_uploaded"] == as_bytes["map_reads"]
    res = {"workload": bench.workload_name(w), "rounds": args.rounds, "rows_identical": identical,
           "mapped_reads": sum(1 for x in rows["map_device"] if x.mapped), "gpu": info_before,
           "gpu_after": info_after, "timing": "device stopwatch (CUDA events on the library stream) per call, "
           "median over the rounds; wall_ms: host clock around the call"}
    for name, t in times.items():
        ms = statistics.median(t["ms"])
        res[name] = {"ms": round(ms, 3), "wall_ms": round(statistics.median(t["wall_ms"]), 3),
                     "ms_all": [round(x, 3) for x in t["ms"]], "samples": t["samples"],
                     "samples_per_s": t["samples"] / (ms / 1000.0), "h2d_bytes": t["h2d_bytes"]}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    m.close()
    if not identical:
        print("device_input_time: the three paths returned different rows", file=sys.stderr)
        sys.exit(1)


if __name__ == "__main__":
    main()
