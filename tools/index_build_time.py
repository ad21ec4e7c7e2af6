#!/usr/bin/env python
"""Wall time of the device point-cloud / index build (smb_point_cloud_build, smb_index_build,
smb_point_cloud_build_part) per stage, against the host build (smbh_build_point_cloud_alloc /
smbh_build_point_cloud_part) on the same box.  Prints one JSON line (and writes it to --out).

Cases (synthetic uniform references, smbh_sim_reference):
  12m   12 Mbp in 16 contigs: device cloud, device index, host cloud
  400m  400 Mbp in 16 contigs: device cloud, device index, host cloud
  3g    3.1 Gbp in 24 contigs, rank 0's part at world 8: device only (the host takes minutes)
Device numbers: one warm-up call, then the median of --runs calls; per-stage CUDA-event ms from
smb_index_build_stats of the median call.  Host numbers: median of --host-runs calls (400m: one).
The card's name, power limit and SM clocks are read before and after the timed calls."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CASES = {
    "12m": (12_000_000, 16, None),
    "400m": (400_000_000, 16, None),
    "3g": (3_100_000_000, 24, 8),
}


def gpu_info(device):
    if not shutil.which("nvidia-smi"):
        return {"nvidia_smi": "unavailable"}
    q = "name,power.limit,clocks.sm,clocks.max.sm,temperature.gpu"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", str(device)],
                         capture_output=True, text=True).stdout.strip()
    return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))


def lengths_of(total, n):
    base = total // n
    return [base + (1 if i < total - base * n else 0) for i in range(n)]


def timed(fn, runs):
    walls, stats = [], []
    for _ in range(runs):
        t0 = time.perf_counter()
        st = fn()
        walls.append(time.perf_counter() - t0)
        stats.append(st)
    k = sorted(range(runs), key=lambda i: walls[i])[runs // 2]
    return {"wall_s": walls[k], "wall_s_all": walls, "stages_ms": stats[k]}


def stage_ms(m):
    st = m.build_stats()
    return {k: round(v, 3) for k, v in st.items() if k.startswith("ms_")} | {
        k: st[k] for k in ("points", "tiles", "tiles_rewalked", "tiles_unconverged", "tiles_redone", "tile",
                          "strands", "strands_serial_mean")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="12m,400m,3g")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--host-runs", type=int, default=3)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from sigmap_b200 import host as H
    from sigmap_b200.mapper import Mapper
    from sigmap_b200.shard import assign_contigs
    model = H.load_pore_model()
    lv = model[0]
    res = {"tool": "index_build_time", "gpu_before": gpu_info(a.device), "host_cores": os.cpu_count(),
           "runs": a.runs, "cases": {}}
    m = Mapper(a.device)
    for name in a.cases.split(","):
        total, n_contigs, world = CASES[name]
        t0 = time.perf_counter()
        ref = H.sim_reference(17, lengths_of(total, n_contigs))
        case = {"bases": total, "contigs": n_contigs, "sim_s": round(time.perf_counter() - t0, 2)}
        if world is None:
            def dev_cloud():
                pos, val = m.point_cloud(ref, lv)
                return stage_ms(m) | {"points_returned": len(pos)}

            def dev_index():
                m.build_index(ref, lv)
                return stage_ms(m)
            dev_cloud()  # warm-up
            case["device_cloud"] = timed(dev_cloud, a.runs)
            case["device_index"] = timed(dev_index, a.runs)
            host_runs = a.host_runs if total < 100_000_000 else 1

            def host_cloud():
                pos, _ = H.build_point_cloud(ref, lv)
                return {"points": len(pos)}
            case["host_cloud"] = timed(host_cloud, host_runs)
            case["host_cloud"]["runs"] = host_runs
            case["same_points"] = case["host_cloud"]["stages_ms"]["points"] == case["device_cloud"]["stages_ms"]["points"]
            case["speedup_cloud"] = round(case["host_cloud"]["wall_s"] / case["device_cloud"]["wall_s"], 1)
            dev_ms = sum(v for k, v in case["device_cloud"]["stages_ms"].items() if k.startswith("ms_"))
            case["speedup_device_stages"] = round(case["host_cloud"]["wall_s"] * 1e3 / dev_ms, 1)
        else:
            owner = assign_contigs(ref.lengths, world)
            case["world"], case["rank"] = world, 0

            def dev_part():
                p = m.point_cloud_part(ref, lv, owner, 0)
                try:
                    n_values = int(p.c.n_values)
                finally:
                    p.close()
                return stage_ms(m) | {"part_values": n_values}
            dev_part()  # warm-up
            case["device_part"] = timed(dev_part, a.runs)
        res["cases"][name] = case
        del ref
        print(json.dumps({name: case}), file=sys.stderr, flush=True)
    m.close()
    res["gpu_after"] = gpu_info(a.device)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
