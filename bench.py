#!/usr/bin/env python
"""bench.py -- raw samples/s mapped by the B200 hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU path
    python bench.py ... --dump-outputs DIR     # + the rows of the last timed step as DIR/*.npy

Workload at N=1 = BASELINE.json configs[1] ("c2"): E. coli-sized 4.6 Mbp synthetic reference,
20 000 simulated reads (R9.4 6-mer model, noise 1.0), full-read mapping (every chunk of every
read is consumed).  One "step" = one pass of the whole hot path over that read batch.  The N=1
line also carries a `config3` object: BASELINE.json configs[2] ("c3") on the same GPU.
N>1 (torchrun, one rank per GPU) = configs[2], the configuration BASELINE.json quotes at
1/2/4/8 GPUs: yeast-sized 12 Mbp x 16 contigs, 100 000 reads with the reference's default stop
rules, the reads split over the ranks (STRONG scaling: the job is fixed), index replicated, no
data-path collective.  The single-GPU figure of the same job is `config3.value` of the N=1 line.

value  = samples mapped / time with the raw int16 reads already resident in HBM
e2e    = the same through smb_map_reads() with pinned HOST buffers (H2D + D2H inside)
concordance = PAF rows of the CUDA path against the unmodified reference binary on the same
         reads (north_star: >= 99.5 %); the bench exits non-zero below that
Times are CUDA-event times on the library's stream, max over ranks.
"""
import argparse
import json
import os
import re
import shutil
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FULL_READ_CLI = ["--max-num-chunks", "100000", "--stop-mapping", "1e30", "--stop-mapping-mean",
                 "1e30", "--min-num-anchors", "2000000000"]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="auto", choices=["auto", "c2", "c3"],
                    help="auto = c2 on one GPU, c3 on several; explicit --ref-bp/--contigs/--reads/--mode override")
    ap.add_argument("--ref-bp", type=int, default=None)
    ap.add_argument("--contigs", type=int, default=None)
    ap.add_argument("--reads", type=int, default=None,
                    help="c2: reads per GPU (weak scaling); c3: reads of the whole job (strong scaling)")
    ap.add_argument("--noise", type=float, default=1.0)
    ap.add_argument("--mode", default=None, choices=["full", "default"],
                    help="full = full-read mapping (configs[1]); default = reference stop rules")
    ap.add_argument("--cpu-sample-reads", type=int, default=0,
                    help="reads the CPU reference maps beside the GPU (0 = max(1500, 50 x host cores))")
    ap.add_argument("--ref-step-reads", type=int, default=0,
                    help="--impl reference: reads per step (0 = max(50 x host cores, min(1500, 20000 / steps)))")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config3", action="store_true", help="N=1: skip the config 3 leg")
    ap.add_argument("--c3-steps", type=int, default=None, help="N=1: timed steps of the config 3 leg (default: --steps)")
    ap.add_argument("--channels", type=int, default=512, help="read-until leg: concurrent channels")
    ap.add_argument("--stream-rounds", type=int, default=24, help="read-until leg: timed rounds (0 = skip)")
    ap.add_argument("--shard", default="reads", choices=["reads", "contigs"],
                    help="N>1: reads = every rank maps its own reads against a replicated index "
                         "(default, weak scaling); contigs = the index is partitioned by contig, every "
                         "rank maps every read, NCCL merges the chains (SURVEY 8e mode 2, strong scaling)")
    ap.add_argument("--seed", type=int, default=20251017)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the rows the last timed step returned as DIR/<field>.npy (config 3 leg: "
                         "DIR/config3_<field>.npy), rank 0 only")
    args = ap.parse_args()
    if args.steps < 1 or (args.c3_steps is not None and args.c3_steps < 1):
        ap.error("--steps and --c3-steps must be at least 1")
    return resolve_workload(args, int(os.environ.get("WORLD_SIZE", "1")))


WORKLOADS = {
    # BASELINE.json configs[1]
    "c2": dict(ref_bp=4_600_000, contigs=1, reads=20000, mode="full", scaling="weak"),
    # BASELINE.json configs[2]
    "c3": dict(ref_bp=12_000_000, contigs=16, reads=100000, mode="default", scaling="strong"),
}


def resolve_workload(args, world):
    name = args.workload
    if name == "auto":
        name = "c2" if world == 1 else "c3"
    if args.shard == "contigs":
        name = "c2" if args.workload == "auto" else name
    w = WORKLOADS[name]
    args.workload = name
    for k in ("ref_bp", "contigs", "reads", "mode"):
        if getattr(args, k) is None:
            setattr(args, k, w[k])
    args.scaling = "strong" if (w["scaling"] == "strong" or args.shard == "contigs") else "weak"
    cores = os.cpu_count() or 1
    if args.cpu_sample_reads <= 0:
        args.cpu_sample_reads = max(1500, 50 * cores)
    if args.ref_step_reads <= 0:
        # the reference arm: every step a bounded sample, at least 50 reads per host thread (fewer
        # starve the reference's taskloop) and sized so that --steps K ends within a few minutes
        args.ref_step_reads = max(50 * cores, min(1500, 20000 // max(args.steps, 1)))
    return args


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.proc = None
        self.lines = []

    def start(self):
        if not shutil.which("nvidia-smi"):
            return
        self.proc = subprocess.Popen(
            ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
             "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        self.t = threading.Thread(target=self._read, daemon=True)
        self.t.start()

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        # "under load": samples at or above the median (the sampler also sees idle gaps)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
    return rank, world, local, dist


def build_workload(args, rank, need_cloud=True):
    from sigmap_b200 import host as H
    model = H.load_pore_model()
    per = args.ref_bp // args.contigs
    ref = H.sim_reference(args.seed, [per] * args.contigs)
    pos, val = H.build_point_cloud(ref, model[0]) if need_cloud else (None, None)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.shard == "contigs":          # contig shards all see the same reads
        first, count = 0, args.reads
    elif args.scaling == "strong":       # the job's reads, split over the ranks
        first = rank * args.reads // world
        count = (rank + 1) * args.reads // world - first
    else:                                # weak: every rank its own reads
        first, count = rank * args.reads, args.reads
    reads = H.sim_reads(args.seed + 1, ref, count, first_read=first, noise=args.noise, model=model)
    return H, model, ref, pos, val, reads


def workload_name(args):
    per = "reads/GPU" if args.scaling == "weak" else "reads in the job"
    return (f"{args.ref_bp / 1e6:.1f} Mbp synthetic reference x{args.contigs} contig(s), "
            f"{args.reads} simulated {per} (R9.4 6-mer model, noise {args.noise}), "
            f"{'full-read' if args.mode == 'full' else 'default stop rules'} mapping")


# ------------------------------------------------------------------ reference arm helpers
def ref_prepare(args, H, ref, reads, n_sample, workdir):
    """FASTA + reference-built index (.pt/.si) + a BLOW5 holding the first n_sample reads."""
    from oracle.oracle import REF_BIN
    fasta = os.path.join(workdir, "ref.fa")
    ref.write_fasta(fasta)
    prefix = os.path.join(workdir, "idx")
    t0 = time.time()
    r = subprocess.run([REF_BIN, "-i", "-r", fasta, "-p", H.MODEL_PATH, "-o", prefix],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("reference index build failed: " + r.stderr[-400:])
    sig = os.path.join(workdir, "sig")
    os.makedirs(sig, exist_ok=True)
    n = min(n_sample, reads.n)
    sub = H.ReadSet(reads.names[:n], reads.raw[:int(reads.read_off[n])], reads.read_off[:n + 1],
                    H.DIGITISATION, H.RANGE, H.OFFSET)
    sub.write_blow5(os.path.join(sig, "sample.blow5"))
    return fasta, prefix, sig, n, time.time() - t0


def ref_map_once(args, H, fasta, prefix, sig, workdir, threads):
    from oracle.oracle import REF_BIN
    out = os.path.join(workdir, "ref.paf")
    cmd = [REF_BIN, "-m", "-r", fasta, "-p", H.MODEL_PATH, "-x", prefix, "-s", sig, "-o", out,
           "-t", str(threads)]
    if args.mode == "full":
        cmd += FULL_READ_CLI
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("reference mapping failed: " + r.stderr[-400:])
    m = re.search(r"Finished mapping in ([0-9.eE+-]+)", r.stderr)
    secs = float(m.group(1))
    samples = 0
    for line in open(out):
        ci = re.search(r"ci:i:(\d+)", line)
        sl = re.search(r"sl:i:(\d+)", line)
        if ci and sl and int(sl.group(1)) >= 4000:
            samples += int(ci.group(1)) * 4000
    return samples, secs


def run_reference(args):
    """The reference's own CPU implementation of the path on this box's host cores (all of them),
    on the arm's workload: every step maps the first --ref-step-reads reads of the job."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle.oracle import Ref
    if not Ref.available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref was not built"}))
        return
    n_step = max(args.ref_step_reads, 1)
    H, model, ref, pos, val, reads = build_workload(
        argparse.Namespace(**{**vars(args), "reads": n_step, "scaling": "weak", "shard": "reads"}), 0)
    threads = os.cpu_count() or 1
    workdir = tempfile.mkdtemp(prefix="sigmap_ref_")
    # a CPU run has no clocks to warm: one warm-up pass (page cache, index load) is all it needs
    warm = min(args.warmup, 1)
    try:
        fasta, prefix, sig, n, t_idx = ref_prepare(args, H, ref, reads, n_step, workdir)
        for _ in range(warm):
            ref_map_once(args, H, fasta, prefix, sig, workdir, threads)
        tot_s, tot_t = 0, 0.0
        for _ in range(args.steps):
            s, t = ref_map_once(args, H, fasta, prefix, sig, workdir, threads)
            tot_s += s
            tot_t += t
    finally:
        shutil.rmtree(workdir, ignore_errors=True)
    value = tot_s / tot_t
    sample = (f"first {n} reads of the workload per step, oracle/_ref/sigmap_ref -m -t {threads} "
              f"(the unmodified reference, strict-FP build without -march=native: the parity pin; "
              f"map phase only, 'Finished mapping in'; index build {t_idx:.0f} s not timed)")
    print(json.dumps({
        "impl": "reference", "metric": "raw samples/sec mapped", "value": value, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": warm,
        "ms_per_step": 1000.0 * tot_t / max(args.steps, 1), "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args), "sample_reads_per_step": n},
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": threads, "kind": "reference",
                         "sample": sample},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def reference_concordance(args, H, ref, reads, rows, mapper, n_sample):
    """Map the first n_sample reads with the unmodified reference binary on this box's cores and
    compare its PAF with the CUDA path's rows of the same reads (north_star: same decision,
    contig, strand, positions within 10 bp).  -> (cpu_baseline dict, concordance dict)"""
    from oracle.oracle import Ref
    from sigmap_b200 import paf_eval
    if not Ref.available():
        return ({"value": None, "unit": "samples/s", "cores": 0, "kind": "reference",
                 "sample": "oracle/_ref not built on this box"}, None)
    threads = os.cpu_count() or 1
    workdir = tempfile.mkdtemp(prefix="sigmap_cpu_")
    try:
        fasta, prefix, sig, n, t_idx = ref_prepare(args, H, ref, reads, n_sample, workdir)
        s, t = ref_map_once(args, H, fasta, prefix, sig, workdir, threads)
        ref_rows = paf_eval.read_paf(os.path.join(workdir, "ref.paf"))
    finally:
        shutil.rmtree(workdir, ignore_errors=True)
    sub = H.ReadSet(reads.names[:n], reads.raw[:int(reads.read_off[n])], reads.read_off[:n + 1],
                    H.DIGITISATION, H.RANGE, H.OFFSET)
    gpu_lines = mapper.paf_lines(sub, rows[:n], ref.names)
    res = paf_eval.concordance(ref_rows, paf_eval.read_paf(gpu_lines))
    gpu_rows = paf_eval.read_paf(gpu_lines)
    same_decision = sum(1 for k, a in ref_rows.items() if k in gpu_rows and a.mapped == gpu_rows[k].mapped and
                        (not a.mapped or (a.contig == gpu_rows[k].contig and a.strand == gpu_rows[k].strand)))
    flagged = sum(1 for m in rows[:n] if m.flags & 1)
    conc = {"reads": res["reads"], "same_decision": same_decision, "within_10bp": res["concordant"],
            "identical_rows": res["identical_rows"], "pct": 100.0 * res["fraction"],
            "reads_with_capped_query": flagged,
            "against": f"oracle/_ref/sigmap_ref -m -t {threads} on the first {n} reads of the workload",
            "criterion": "same mapped/unmapped decision, contig and strand; target start and end within 10 bp"}
    cpu = {"value": s / t, "unit": "samples/s", "cores": threads, "kind": "reference",
           "sample": f"first {n} reads of the workload, oracle/_ref/sigmap_ref -m -t {threads} (unmodified reference, "
                     f"strict-FP build without -march=native), map phase only ({t:.1f} s; index build {t_idx:.0f} s not timed)"}
    return cpu, conc


# ------------------------------------------------------------------ read-until latency leg
def stream_latency(mapper, reads, n_channels, rounds, warm=3):
    """BASELINE.json's second metric (configs[3]): 512 concurrent channels, one 4 000-sample chunk
    per channel per round, default stop rules, finished channels refilled with the next read.
    Latency of a chunk = duration of the smb_stream_round call that carries it (host samples in,
    stop decision out, copies included), host clock; p50 over all chunks of the timed rounds."""
    import numpy as np
    from sigmap_b200.mapper import default_params
    if rounds <= 0 or reads.n == 0:
        return None
    chunk = 4000
    mapper.stream_open(n_channels, default_params())
    cur, at, nxt = [0] * n_channels, [0] * n_channels, 0

    def assign(ch):
        nonlocal nxt
        for _ in range(reads.n):  # next read holding at least one chunk
            r = nxt % reads.n
            nxt += 1
            if int(reads.read_off[r + 1] - reads.read_off[r]) >= chunk:
                break
        cur[ch], at[ch] = r, 0
        mapper.stream_begin_read(ch, float(reads.digitisation[r]), float(reads.range[r]),
                                 float(reads.offset[r]))

    for ch in range(n_channels):
        assign(ch)
    channels = np.arange(n_channels, dtype=np.uint32)
    off = (np.arange(n_channels + 1, dtype=np.uint64) * chunk).astype(np.uint32)
    samples = np.zeros(n_channels * chunk, np.int16)
    lat, stops, detail = [], 0, []
    for rd in range(warm + rounds):
        for ch in range(n_channels):
            o = int(reads.read_off[cur[ch]]) + at[ch]
            samples[ch * chunk:(ch + 1) * chunk] = reads.raw[o:o + chunk]
        before = mapper.stats()
        t0 = time.perf_counter()
        dec, _ = mapper.stream_round_arrays(channels, samples, off)
        dt = time.perf_counter() - t0
        if rd >= warm:
            lat.append(dt * 1000.0)
            stops += int(dec.sum())
            after = mapper.stats()
            detail.append({"round": rd - warm, "ms": round(dt * 1000.0, 3),
                           **{k: round(after[k] - before[k], 3) for k in
                              ("ms_events", "ms_search", "ms_sort", "ms_chain", "ms_stream_stage", "steps", "chunks", "anchors")}})
        for ch in range(n_channels):
            at[ch] += chunk
            r = cur[ch]
            if dec[ch] or at[ch] + chunk > int(reads.read_off[r + 1] - reads.read_off[r]):
                assign(ch)
    mapper.stream_close()
    lat.sort()
    q = lambda f: lat[min(len(lat) - 1, int(f * len(lat)))]
    return {"metric": "per-chunk latency, read-until mode", "unit": "ms", "p50": q(0.5), "p90": q(0.9),
            "max": lat[-1], "channels": n_channels, "rounds": rounds, "chunks": rounds * n_channels,
            "stop_decisions": stops, "chunk_samples": chunk,
            "slowest_rounds": sorted(detail, key=lambda d: -d["ms"])[:3],
            "samples_per_s": rounds * n_channels * chunk / (sum(lat) / 1000.0),
            "timed": "smb_stream_round call, host buffers in -> decisions out (host clock)"}


# ------------------------------------------------------------------ output dump
DUMP_BYTES_PER_LEG = 32 << 20   # two legs at N=1: at most 64 MB in all


def dump_rows(rows, directory, prefix, seed):
    """The smb_mapping rows of a mapping call, one DIR/<prefix><field>.npy per field (float32 for
    the float fields, float64 for the integer ones: exact) and <prefix>read_index.npy, the read
    each row belongs to.  Above DUMP_BYTES_PER_LEG a fixed sample of the rows, drawn from --seed."""
    import ctypes as C
    from sigmap_b200 import _ffi as F
    fields = [(n, t is C.c_float) for n, t in F.Mapping._fields_]
    dt = np.dtype([(n, "<f4" if flt else "<u4") for n, flt in fields])
    assert dt.itemsize == C.sizeof(F.Mapping)
    n = len(rows)
    row_bytes = 8 + sum(4 if flt else 8 for _, flt in fields)
    keep = np.arange(n)
    if n * row_bytes > DUMP_BYTES_PER_LEG:
        keep = np.sort(np.random.default_rng(seed).choice(n, DUMP_BYTES_PER_LEG // row_bytes, replace=False))
    a = np.frombuffer(b"".join(bytes(rows[int(i)]) for i in keep), dt)
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, prefix + "read_index.npy"), keep.astype(np.float64))
    for name, flt in fields:
        np.save(os.path.join(directory, prefix + name + ".npy"), a[name].astype(np.float32 if flt else np.float64))


# ------------------------------------------------------------------ our arm
def measure(args, rank, world, local, dist, light=False):
    """One workload on this rank's GPU: device-resident leg, end-to-end leg, (read-until leg),
    roofline of the dominant kernel, CPU reference + concordance beside it.  `light`: the config 3
    leg of an N=1 run (fewer steps, no read-until leg)."""
    import torch
    from sigmap_b200.mapper import Mapper, default_params, full_read_params

    steps = (args.c3_steps or args.steps) if light else args.steps
    warmup = min(args.warmup, 1) if light else args.warmup
    t_setup = time.time()
    by_contig = args.shard == "contigs" and world > 1
    replicate = world > 1 and not by_contig
    # read-sharded: only rank 0 builds the point cloud and the device index; the others receive the
    # index over NVLink (one ncclBroadcast on the library's own communicator)
    # contig-sharded: a rank only ever builds its own part of the cloud (the genome-scale path)
    H, model, ref, pos, val, reads = build_workload(args, rank, need_cloud=not by_contig and (not replicate or rank == 0))
    mapper = Mapper(local)  # raises if there is no CUDA device: no fallback
    t_bcast = None
    if by_contig:
        from sigmap_b200 import shard
        shard.nccl_join(mapper, dist)  # the library's own NCCL communicator, on its own stream
        part = H.build_point_cloud_part(ref, model[0], shard.assign_contigs(ref.lengths, world), rank)
        mapper.set_index_part(part, ref.n)
        part.close()
    elif replicate:
        from sigmap_b200 import shard
        shard.nccl_join(mapper, dist)
        if rank == 0:
            mapper.set_index(pos, val)
            mapper.set_contigs(ref.lengths)
        dist.barrier()
        t_bcast = time.time()
        mapper.broadcast_index(0)
        t_bcast = time.time() - t_bcast
    else:
        mapper.set_index(pos, val)
    mapper.set_contigs(ref.lengths)
    n_points = int(mapper.num_points)
    params = full_read_params() if args.mode == "full" else default_params()
    # pinned host staging of the raw reads (e2e leg copies from here every step)
    pinned = torch.empty(len(reads.raw), dtype=torch.int16, pin_memory=True)
    pinned.numpy()[:] = reads.raw
    reads.raw = pinned.numpy()
    t_setup = time.time() - t_setup

    def barrier():
        torch.cuda.synchronize(local)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(local)

    def reduce(x, op):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local}")
        dist.all_reduce(t, op=op)
        return float(t.item())

    max_over_ranks = lambda x: reduce(x, dist.ReduceOp.MAX) if dist is not None else x
    sum_over_ranks = lambda x: reduce(x, dist.ReduceOp.SUM) if dist is not None else x

    # ---- device-resident leg
    mapper.upload_reads(reads)
    for _ in range(warmup):
        rows = mapper.map_uploaded(params)
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    mapper.stats_reset()
    mapper.timer_start()
    t_wall = time.time()
    for _ in range(steps):
        rows = mapper.map_uploaded(params)
    ms = mapper.timer_stop()
    t_wall = time.time() - t_wall
    barrier()
    st = mapper.stats()
    clocks = sampler.stop()
    ms = max_over_ranks(ms)
    # contig shards all map the same reads: the job's samples are one rank's, not the sum
    samples_total = float(st["samples"]) if by_contig else sum_over_ranks(float(st["samples"]))
    value = samples_total / (ms / 1000.0)
    n_mapped = sum(1 for m in rows if m.mapped)
    # concordance with the simulation truth (sanity, not a parity claim)
    ok = 0
    for r, m in enumerate(rows):
        c, s, e, plus = (int(v) for v in reads.truth[r])
        if m.mapped and m.contig == c and m.strand_plus == plus and m.t_start < e + 50 and \
                m.t_start + m.frag_len > s - 50:
            ok += 1
    n_mapped, ok = int(sum_over_ranks(n_mapped)), int(sum_over_ranks(ok))

    # ---- end-to-end leg: host buffers in, rows out, copies inside the timed region, all steps
    mapper.map_reads(reads, params)  # one warm-up
    barrier()
    mapper.stats_reset()
    mapper.timer_start()
    for _ in range(steps):
        mapper.map_reads(reads, params)
    ms_e2e = mapper.timer_stop()
    barrier()
    st2 = mapper.stats()
    ms_e2e = max_over_ranks(ms_e2e)
    e2e_samples = float(st2["samples"]) if by_contig else sum_over_ranks(float(st2["samples"]))
    e2e_value = e2e_samples / (ms_e2e / 1000.0)

    # ---- read-until leg (per-chunk latency, 512 channels), rank 0 only
    latency = None
    if rank == 0 and args.stream_rounds > 0 and not by_contig and not light:
        latency = stream_latency(mapper, reads, args.channels, args.stream_rounds)
    barrier()

    # ---- roofline of the dominant kernel (radius search), live CUDA-event timing
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    L = max(st["search_launches"], 1)
    alg_bytes = (24.0 * st["queries"] + 44.0 * st["hits"]) / L   # SURVEY.md 8(d) per-unit figures
    dur_s = st["ms_search"] / 1000.0 / L
    achieved = alg_bytes / dur_s / 1e9 if dur_s > 0 else 0.0
    traffic, ncu_note = None, None
    tpath = os.path.join(ROOT, "profiles", "search_traffic.json")
    if os.path.exists(tpath) and args.workload == "c2":  # one ncu --set full capture of a whole c2 step
        tj = json.load(open(tpath))
        traffic = tj.get("dram_bytes_per_launch")
        ncu_note = {"limiter": tj.get("limiter"), **(tj.get("ncu") or {})}
    pipeline_bytes = (2.0 * st["samples"] + 8.0 * st["events"] + 24.0 * st["queries"] +
                      44.0 * st["hits"] + 44.0 * st["anchors"])
    per_gpu = 1 if by_contig else max(world, 1)
    pipe_gbps = sum_over_ranks(pipeline_bytes) / (ms / 1000.0) / 1e9 / max(world, 1) if not by_contig else \
        pipeline_bytes / (ms / 1000.0) / 1e9
    counters = {k: int(sum_over_ranks(float(st[k])) // max(steps, 1)) for k in
                ("samples", "events", "queries", "hits", "anchors", "capped_queries", "chunks", "steps", "linked", "pending",
                 "seg_sort_steps", "part_sort_steps", "overflow_queries", "sync_points")}

    out = {
        "metric": "raw samples/sec mapped", "value": value, "unit": "samples/s",
        "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": ms / max(steps, 1), "higher_is_better": True,
        "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args), "baseline_config": {"c2": "configs[1]", "c3": "configs[2]"}[args.workload],
                   "l2": "inputs larger than L2 (raw reads + index)",
                   "index_points": n_points, "reads_this_rank": int(reads.n),
                   "index_broadcast_s": t_bcast,
                   "parallelism": (f"index sharded by contig x{world}, every rank maps every read, "
                                   f"{int(st['exchanges'])} NCCL collectives per rank in the timed region"
                                   if by_contig else
                                   (f"the job's reads split over {world} rank(s), index built on rank 0 and replicated with one "
                                    f"ncclBroadcast, no data-path collective"
                                    if args.scaling == "strong" else f"read-sharded x{world}, index replicated"))},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "samples/s",
                "h2d_bytes_per_step": int(st2["h2d_bytes"] // steps),
                "d2h_bytes_per_step": int(st2["d2h_bytes"] // steps), "steps": steps},
        "gpu_launches": int(st["launches"]),
        "roofline": {"bound": "hbm", "kernel": "k_search_lean (+ k_radius_search for overflow queries)",
                     "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes,
                     "avg_launch_ms": dur_s * 1000.0, "launches": int(st["search_launches"]),
                     "ncu": ncu_note},
        "pipeline": {"algorithmic_GBps": pipe_gbps, "frac_of_hbm": pipe_gbps / peak,
                     "kernel_ms_per_step": {k: st[k] / max(steps, 1) for k in
                                            ("ms_filter", "ms_events", "ms_search", "ms_sort", "ms_chain")},
                     "wall_ms_per_step": 1000.0 * t_wall / max(steps, 1),
                     "counters_per_step": counters},
        "latency": latency,
        "mapped_reads": n_mapped, "truth_concordant_reads": ok, "setup_s": t_setup,
    }

    # ---- CPU reference beside it (rank 0): throughput on a bounded sample at N=1, and the PAF
    # concordance of the CUDA rows with the reference's on those reads at every N
    if rank == 0 and not args.no_cpu_baseline:
        n_sample = args.cpu_sample_reads if world == 1 else min(args.cpu_sample_reads, 300)
        if light:
            n_sample = min(n_sample, 600)
        try:
            cpu, conc = reference_concordance(args, H, ref, reads, rows, mapper, min(n_sample, reads.n))
        except Exception as e:  # the baseline is reported, never fatal
            cpu, conc = ({"value": None, "unit": "samples/s", "cores": 0, "kind": "reference",
                          "sample": f"failed: {e}"}, None)
        if world == 1:
            out["cpu_baseline"] = cpu
        out["concordance"] = conc
    if rank == 0 and args.dump_outputs:
        dump_rows(rows, args.dump_outputs, "config3_" if light else "", args.seed)
    mapper.close()
    del pinned
    return out


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return
    # torchrun pins OMP_NUM_THREADS=1 in every worker; the host-side setup (simulator, point
    # cloud) is OpenMP code and would crawl: give each rank its share of the cores instead
    w_env = int(os.environ.get("WORLD_SIZE", "1"))
    if w_env > 1 and os.environ.get("OMP_NUM_THREADS", "1") == "1":
        os.environ["OMP_NUM_THREADS"] = str(max(1, (os.cpu_count() or 1) // w_env))
    rank, world, local, dist = dist_setup(args.gpus)
    out = measure(args, rank, world, local, dist)
    # N=1: the configuration BASELINE.json quotes at 1/2/4/8 GPUs, on this one GPU (the
    # single-GPU point of the strong-scaling curve the N>1 lines continue)
    if world == 1 and args.workload == "c2" and not args.no_config3:
        a3 = argparse.Namespace(**{**vars(args), "workload": "c3", "ref_bp": None, "contigs": None,
                                   "reads": None, "mode": None})
        a3 = resolve_workload(a3, 2)
        a3.workload = "c3"
        c3 = measure(a3, rank, world, local, dist, light=True)
        out["config3"] = {k: c3[k] for k in ("value", "unit", "ms_per_step", "steps", "scaling", "config", "e2e",
                                             "roofline", "pipeline", "mapped_reads", "truth_concordant_reads",
                                             "concordance", "setup_s") if k in c3}
    if rank == 0:
        print(json.dumps(out))
    if dist is not None:
        dist.destroy_process_group()
    bad = [c for c in (out.get("concordance"), (out.get("config3") or {}).get("concordance"))
           if c and c["pct"] < 99.5]
    if rank == 0 and bad:
        print(f"bench: PAF concordance with the reference below 99.5 %: {bad}", file=sys.stderr)
        sys.exit(1)


if __name__ == "__main__":
    main()
