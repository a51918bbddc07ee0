#!/usr/bin/env python
"""bench.py -- reads SW-scored/sec of the per-locus read-scoring path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host cores

A *step* is one pass of the whole hot path (CB lookup -> 2x Smith-Waterman per pair -> call -> count
matrix -> triplets) over one synthetic shard of a BASELINE.json shape (default config3: 100k SNV loci x 50k
barcodes, 150 bp reads, 50x, consensus mode -- the shape the metric is quoted on); the unit is the (read, locus)
pair that reaches the aligner (main.rs:896-930).  With N GPUs the loci shard across ranks with no data-path
collective: `--scaling weak` (default) gives every rank its own shard of the shape, `--scaling strong` splits the
shape's loci over the ranks.  The finished triplets are assembled over NCCL inside the timed region, by default on
the rank that writes the matrix (`--gather root`, ncclSend/Recv) and overlapped with the next step's kernels;
`--gather all` is the allgatherv on every rank.

`value`  : pairs/s with the staged shard already resident in HBM (vtx_submit2_device + vtx_finish_device).
`e2e`    : pairs/s through the host-facing C ABI from pinned HOST buffers (vtx_submit2 + vtx_finish), i.e. with the
           host->device copy of the shard (slim staging layout, ~96 B per candidate) and the device->host copy of the
           triplets in the timed region.  The step's shard is handed over the way a staging producer would: a 1 % shard
           (at least 100 k candidates) first, then shards growing by up to 2x (less when the measured copy/kernel ratio
           asks for it) up to 1/6 of the step, so that every copy hides behind the previous shard's kernels.
`roofline`: the dominant kernel (vtx_k_sw_fold for windows built with --padding >= 96) against the measured HBM
           peak, from CUDA events recorded on the engine's stream inside the library (vtx_last_timing), averaged over
           the timed steps; `roofline.issue_bound` is the same kernel against the ALU-pipe bound that actually binds.
`cpu_baseline`: the oracle's C port of the reference algorithm timed on this box's host cores (bounded sample), with its
           thread scaling and the cgroup CPU quota, so that a CPU-starved box explains itself.

`--dump-outputs DIR` writes the triplets the last timed `value` step returned as float64 .npy files (see dump_outputs),
so that two builds run with the same arguments -- hence the same seeded shard -- can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "reads_sw_scored_per_sec"
UNIT = "pairs/s"


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError(f"must be at least 1, got {v}")
    return v


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=5, help="timed steps of each measured path")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="vartrix_b200", choices=["vartrix_b200", "reference"])
    ap.add_argument("--workload", default="config3", help="synth.CONFIGS key (config3 = the shape the metric is quoted on)")
    ap.add_argument("--loci", type=int, default=0, help="override the shape's number of loci (0 = the config's)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="weak: the shape per GPU; strong: the shape's loci split over the GPUs")
    ap.add_argument("--submits", type=int, default=0, help="device-resident submits per step for `value` (0 = 1, or 4 for shards above 8 M candidates: streamed)")
    ap.add_argument("--gather", default="root", choices=["root", "all"], help="N > 1: triplets to the writer rank (ncclSend/Recv) or to every rank (allgatherv)")
    ap.add_argument("--layout", default="slim", choices=["slim", "v1"], help="staging layout: vtx_batch2 (slim) or vtx_batch")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU time of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--chunks", type=int, default=6, help="staged shards per step on the e2e path (copy/compute overlap); with --growth: largest shard = 1/chunks of the step")
    ap.add_argument("--growth", type=float, default=2.0, help="e2e shards grow geometrically from --first-chunk by this factor (0: equal shards after the first)")
    ap.add_argument("--first-chunk", type=float, default=0.01, help="fraction of the candidates in the first (priming) shard")
    ap.add_argument("--min-shard", type=int, default=100_000, help="e2e shards are not made smaller than this many candidates (per-submit fixed costs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="", help="write the last timed step's triplets to DIR/<name>.npy (one process only)")
    return ap.parse_args(argv)


def dist_env():
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def workload_config(args, rank, world=1):
    import vartrix_b200 as vb
    from vartrix_b200 import dist as vdist
    cfg = dict(vb.synth.CONFIGS[args.workload])
    if args.loci:
        cfg["n_loci"] = args.loci
    if args.scaling == "strong" and world > 1:
        cfg["n_loci"] = max(1, cfg["n_loci"] // world)       # contiguous locus ranges of the one shape (main.rs:250-254)
    return vdist.rank_workload(cfg, rank)      # same barcode list everywhere, own loci/reads, rows offset by rank


def describe(args, cfg, world, info, extra=None):
    per = "per GPU" if args.scaling == "weak" or world == 1 else f"per GPU ({cfg['n_loci'] * world} in total, split over {world})"
    d = {
        "workload": f"{args.workload}: synthetic {cfg['n_loci']} {cfg['kind'].upper()} loci x {cfg['n_barcodes']} barcodes {per}, "
                    f"{info['read_len']} bp reads, {info['depth']}x depth, {cfg['scoring_method']} mode"
                    + (", --umi" if cfg.get("umi") else ""),
        "loci_per_gpu": cfg["n_loci"], "barcodes": cfg["n_barcodes"], "pairs_per_gpu": info["n_pairs"],
        "candidates_per_gpu": info["n_cand"], "scoring_method": cfg["scoring_method"], "umi": bool(cfg.get("umi")),
        "parallelism": (f"loci sharded over {world} GPU(s), {args.scaling} scaling; triplets gathered over NCCL "
                        f"({'to rank 0 with ncclSend/Recv' if args.gather == 'root' else 'allgatherv on every rank'}), overlapped with the next step; "
                        f"on the e2e path every rank copies its own row range to its host (h2d/d2h bytes are job totals)") if world > 1 else "1 GPU",
        "l2_policy": "inputs larger than L2 (staged shard >> 126 MB), no explicit flush",
        "staging_layout": "vtx_batch2 (slim)" if args.layout == "slim" else "vtx_batch",
        "e2e_chunks": args.chunks, "e2e_first_chunk_frac": args.first_chunk, "e2e_chunk_growth_cap": args.growth, "host_cores_bound_to_gpu": len(os.sched_getaffinity(0)),
    }
    d.update(extra or {})
    return d


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle's C port of the reference algorithm on the host cores
# ------------------------------------------------------------------------------------------------
def cgroup_cpu_quota():
    """-> cores the cgroup lets this process use (cpu.max quota / period), or None when unlimited / unknown."""
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] == "max":
                    return None
                return float(txt[0]) / float(txt[1])
            q = float(txt[0])
            if q <= 0:
                return None
            return q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        except Exception:
            continue
    return None


def cpu_threads():
    """Threads the CPU arm may use: the affinity mask, capped at twice the cgroup CPU quota when there is one (a box that
    shows 128 logical CPUs but grants 16 cores of quota runs 128 busy threads slower than 32)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    q = cgroup_cpu_quota()
    if q:
        n = max(1, min(n, int(round(2 * q))))
    return n


def pick_growth(h2d_ms, kernel_ms, cap):
    """Largest shard-to-shard growth whose host->device copy still hides behind the previous shard's kernels,
    with 10 % slack, between 1.1 and `cap`."""
    if h2d_ms <= 0 or kernel_ms <= 0:
        return cap
    return float(min(cap, max(1.1, round(0.9 * kernel_ms / h2d_ms, 2))))


def cpu_sample_run(sb, bcs, cfg, n_loci_sample, threads, band_model=False):
    """-> (pairs, seconds) of the oracle on the first n_loci_sample loci of the shard."""
    from oracle import pipeline as P
    sub = sb.shard(0, n_loci_sample)
    ob = P.Batch(**{f: getattr(sub, f) for f in P.Batch.FIELDS}, n_rows=sub.n_rows).normalized()
    obc = P.Barcodes(bcs.keys)
    t0 = time.perf_counter()
    res = P.run_batch(ob, obc, P.MODES[cfg["scoring_method"]], bool(cfg.get("umi")), n_threads=threads, band_model=band_model)
    dt = time.perf_counter() - t0
    return res.metrics["num_scored"], dt


def cpu_baseline(sb, bcs, cfg, info, target_s):
    """The reference algorithm on the host cores: headline = full-matrix SW port on every usable thread; beside it the
    thread-scaling curve, the cgroup quota and the band-model work profile (what bio 0.30.0's band would leave to do)."""
    threads = cpu_threads()
    quota = cgroup_cpu_quota()
    per_locus = max(info["n_pairs"] / sb.n_loci, 1)
    probe_loci = min(sb.n_loci, max(threads * 4, 128))
    pairs, dt = cpu_sample_run(sb, bcs, cfg, probe_loci, threads)
    rate = pairs / max(dt, 1e-9)
    n_loci = int(min(sb.n_loci, max(probe_loci, 0.45 * target_s * rate / per_locus)))
    pairs, dt = cpu_sample_run(sb, bcs, cfg, n_loci, threads)
    value = pairs / dt
    scaling = {}
    try:
        all_threads = len(os.sched_getaffinity(0))
    except Exception:
        all_threads = threads
    for t in sorted({1, 8, 32, threads, all_threads}):
        if t > all_threads:
            continue
        nl = int(min(sb.n_loci, max(t * 4, 0.1 * target_s * (value * t / threads) / per_locus, 32)))
        p, d = cpu_sample_run(sb, bcs, cfg, nl, t)
        scaling[str(t)] = p / d
    best_t = max(scaling, key=lambda k: scaling[k])
    if scaling[best_t] > value:             # the headline is the best the box gives, whatever the thread count
        value, threads = scaling[best_t], int(best_t)
    v1 = scaling.get("1", value / threads)
    eff = value / (v1 * threads) if v1 > 0 else None
    nb = int(min(sb.n_loci, max(threads * 4, 0.25 * target_s * value / per_locus)))
    pb, db = cpu_sample_run(sb, bcs, cfg, nb, threads, band_model=True)
    return {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "value_1thread": v1,
            "thread_scaling_pairs_per_s": scaling, "parallel_efficiency": eff,
            "cores_effective": (value / v1 if v1 > 0 else None), "cgroup_cpu_quota_cores": quota, "os_cpu_count": os.cpu_count(),
            "band_model_value": pb / db,
            "which_is_headline": "value = full-matrix affine local SW (60 300 cells per pair), the port that reproduces the reference's goldens; "
                                 "band_model_value = the same port restricted to the k=6/w=20 band model of bio 0.30.0 (oracle/vtx_oracle.c::vtxo_sw_band_model: "
                                 "seeding + chaining + ~17 k cells per pair), the closer stand-in for the Rust binary's work profile",
            "sample": f"first {n_loci} loci of the shard ({pairs} pairs, {dt:.1f} s); full-matrix SW C port of the reference "
                      f"algorithm (oracle/vtx_oracle.c), static locus chunks like main.rs:250-254, {threads} threads; "
                      f"band model on {pb} pairs in {db:.1f} s; the Rust binary cannot be built here"}


def run_reference(args):
    rank, world, local = dist_env()
    if rank != 0:
        return 0
    import vartrix_b200 as vb
    cfg = workload_config(args, 0)
    # a bounded sample of the same workload per step, sized so the whole run ends within a few minutes
    threads = cpu_threads()
    probe_cfg = dict(cfg); probe_cfg["n_loci"] = max(threads * 16, 256)
    sb, bcs, info = vb.synth.make_shard(**probe_cfg)
    pairs, dt = cpu_sample_run(sb, bcs, cfg, sb.n_loci, threads)
    rate = pairs / dt
    budget_s = 150.0 / max(1, args.steps + args.warmup)
    n_loci = int(min(cfg["n_loci"], max(probe_cfg["n_loci"], min(budget_s, 20.0) * rate / (info["n_pairs"] / sb.n_loci))))
    scfg = dict(cfg); scfg["n_loci"] = n_loci
    sb, bcs, info = vb.synth.make_shard(**scfg)
    for _ in range(args.warmup):
        cpu_sample_run(sb, bcs, cfg, min(sb.n_loci, probe_cfg["n_loci"]), threads)
    t_tot, p_tot = 0.0, 0
    for _ in range(args.steps):
        p, d = cpu_sample_run(sb, bcs, cfg, sb.n_loci, threads)
        t_tot += d; p_tot += p
    value = p_tot / t_tot
    p1, d1 = cpu_sample_run(sb, bcs, cfg, min(sb.n_loci, 160), 1)
    full_cfg = dict(cfg)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t_tot / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "int32", "data": "synthetic", "impl": "reference",
        "config": describe(args, full_cfg, 1, dict(info, n_pairs=info["n_pairs"], n_cand=info["n_cand"])),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "value_1thread": p1 / d1,
                         "cores_effective": value / (p1 / d1), "cgroup_cpu_quota_cores": cgroup_cpu_quota(), "os_cpu_count": os.cpu_count(),
                         "sample": f"{n_loci} loci of the workload shape per step ({info['n_pairs']} pairs); C port of the reference "
                                   f"algorithm (full-matrix SW), {threads} host threads; the Rust binary cannot be built here"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md recipe)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True); self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append([t.strip() for t in ln.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try: self.proc.wait(timeout=2)
        except Exception: self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def triplet_checksum(row, col, val):
    """Order-independent 64-bit checksum of a triplet set (sum of per-entry mixes, wrapping)."""
    with np.errstate(over="ignore"):
        x = (row.astype(np.uint64) * np.uint64(0x9E3779B97F4A7C15)) ^ (col.astype(np.uint64) * np.uint64(0xC2B2AE3D27D4EB4F)) ^ \
            np.ascontiguousarray(val, np.float64).view(np.uint64)
        x ^= x >> np.uint64(29); x *= np.uint64(0xBF58476D1CE4E5B9); x ^= x >> np.uint64(32)
        return int(x.sum(dtype=np.uint64))


DUMP_MAX_ENTRIES = 1 << 20      # 4 float64 arrays of 1 M entries = 32 MB


def dump_outputs(out_dir, res, with_val2):
    """Write `res` (Triplets) to out_dir as float64 .npy files: row, col, val and, when the mode fills a ref matrix, val2,
    each at the same positions -- all of them, or a seeded sample of DUMP_MAX_ENTRIES in triplet order when there are
    more -- plus metrics.npy = [triplets, num_scored, num_not_cell_bc, num_non_umi] of the whole result."""
    os.makedirs(out_dir, exist_ok=True)
    n = len(res.row)
    idx = np.arange(n)
    if n > DUMP_MAX_ENTRIES:
        idx = np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_ENTRIES, replace=False))
    for name in ("row", "col", "val") + (("val2",) if with_val2 else ()):
        np.save(os.path.join(out_dir, f"{name}.npy"), getattr(res, name)[idx].astype(np.float64))
    m = res.metrics
    np.save(os.path.join(out_dir, "metrics.npy"), np.array([n, m["num_scored"], m["num_not_cell_bc"], m["num_non_umi"]], np.float64))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist
    import vartrix_b200 as vb
    from vartrix_b200 import _capi

    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: vartrix_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes the result of one process: run it without torchrun")
    # stdout carries exactly one JSON line: anything native libraries print there (e.g. NCCL's version banner)
    # goes to stderr instead
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local)
    # bind this rank to the CPU cores next to its GPU (NVML affinity) so that pinned staging buffers are allocated
    # on the GPU-local NUMA node; the full affinity mask comes back before the CPU baseline is timed
    full_affinity = os.sched_getaffinity(0)
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByUUID("GPU-" + str(torch.cuda.get_device_properties(local).uuid))
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cores = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1} & full_affinity
        if cores:
            os.sched_setaffinity(0, cores)
    except Exception:
        pass
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    cfg = workload_config(args, rank, world)
    sb, bcs, info = vb.synth.make_shard(**cfg)
    n_pairs = info["n_pairs"]
    use_umi = bool(cfg.get("umi"))
    slim = args.layout == "slim"
    staged = vb.SlimBatch.from_staged(sb, use_umi) if slim else sb
    fields = vb.SlimBatch.ARRAYS if slim else vb.StagedBatch.FIELDS

    stream = torch.cuda.Stream()
    eng = vb.Engine(cfg["scoring_method"], umi=use_umi, device=local, stream=stream.cuda_stream, values_only=True)
    eng.set_barcodes(bcs)
    if world > 1:       # ship the NCCL unique id of the engine's own communicator over torch.distributed
        from vartrix_b200 import dist as vdist
        uid = vdist.broadcast_bytes(vb.Engine.comm_unique_id() if rank == 0 else None, 128, device="cuda")
        eng.comm_init(uid, rank, world)
    root = 0 if args.gather == "root" else _capi.GATHER_ALL
    keep_alive = []

    def place(batch, where):
        """C struct of `batch` whose arrays live in pinned host memory ("pinned") or on the device ("cuda")."""
        ptr = {}
        for f in fields:
            a = getattr(batch, f)
            if a is None or a.size == 0:
                continue
            t = torch.from_numpy(a.view(np.uint8).reshape(-1) if a.dtype.itemsize > 1 else a.reshape(-1))
            t = t.pin_memory() if where == "pinned" else t.cuda()
            keep_alive.append(t)
            ptr[f] = t.data_ptr()
        if slim:
            return batch.to_c(ptr)
        cb = batch.to_c()
        for f in fields:
            setattr(cb, f, ptr.get(f))
        return cb

    def submit_host(cb):
        rc = (eng._L.vtx_submit2 if slim else eng._L.vtx_submit)(eng._h, C.byref(cb)); eng._ck(rc, "vtx_submit")

    import ctypes as C
    max_read, max_hap = int(info["read_len"]), int(info["max_hap_len"])
    # `value`: the shard resident in HBM, as one submit or (shards above 8 M candidates, or --submits) streamed in several
    n_sub = args.submits or (4 if info["n_cand"] > 8_000_000 else 1)
    dparts = [place(staged.shard(lo, hi) if n_sub > 1 else staged, "cuda") for lo, hi in vb.shard_bounds(sb.cand_start, n_sub) if hi > lo]

    def submit_dev(cb):
        if slim:
            eng.submit2_device(cb, max_read, max_hap)
        else:
            eng.submit_device(cb, max_read, max_hap)

    pending = [False]

    def gather_step():
        """Start this step's gather behind the previous one (which the kernels of this step overlapped)."""
        if world == 1:
            return
        if pending[0]:
            eng.gather_wait()
        eng.gather_start(root)
        pending[0] = True

    def gather_flush():
        if pending[0]:
            res = eng.gather_wait(); pending[0] = False
            return res
        return None

    def step_device():
        for cb in dparts:
            submit_dev(cb)
        res = eng.finish_device()
        gather_step()
        return res

    # e2e: the staging producer hands the engine self-contained shards in pinned memory; the engine double-buffers them so
    # the copy of shard k+1 overlaps the kernels of shard k
    def stage_e2e_shards(growth):
        parts, nbytes = [], 0
        first = max(args.first_chunk, min(1.0, args.min_shard / max(info["n_cand"], 1)))
        for lo, hi in vb.shard_bounds(sb.cand_start, max(1, args.chunks), first_frac=first, growth=growth):
            if hi <= lo:
                continue
            part = staged.shard(lo, hi)
            parts.append(place(part, "pinned")); nbytes += part.nbytes()
        return parts, nbytes

    def step_e2e():
        for cb in hparts:
            submit_host(cb)
        # vtx_finish streams this rank's triplets into the library's pinned host arrays while later shards compute.
        # With several ranks every rank ends up with its own contiguous row range on its host (rank r writes block r
        # of the .mtx at its offset); the NCCL gather still assembles the whole matrix on the writer's GPU.
        out = eng.finish(copy=False)
        gather_step()
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, sampler=None):
        sw_ms, launches = [], 0
        barrier()
        if sampler: sampler.start()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        last = None
        for _ in range(steps):
            last = fn()
            t = eng.timing(); sw_ms.append(t["sw_ms"]); launches += t["total_launches"]
        gather_flush()                      # the last step's gather belongs to the timed region
        e1.record(stream)
        barrier()
        wall = time.perf_counter() - t0
        clocks = sampler.stop() if sampler else None
        dev_ms = e0.elapsed_time(e1)
        # steps end with a host-visible result (vtx_finish* synchronises the engine stream, gather_flush the communication
        # stream), so the wall clock between the two barriers bounds the device time from above: report the larger
        ms = max(dev_ms, wall * 1e3)
        if world > 1:
            tt = torch.tensor([ms], device="cuda", dtype=torch.float64); dist.all_reduce(tt, op=dist.ReduceOp.MAX); ms = float(tt.item())
        return ms, sw_ms, launches, last, clocks

    for _ in range(max(args.warmup, 3)):
        step_device()
    gather_flush()
    sampler = ClockSampler(local) if rank == 0 else None
    ms, sw_ms, launches, last, clocks = timed(step_device, args.steps, sampler)
    if args.dump_outputs:       # before the e2e steps below reuse the engine's result arrays
        dump_outputs(args.dump_outputs, eng.fetch(last), cfg["scoring_method"] == "coverage")
    total_pairs = n_pairs * world
    if world > 1:
        tp = torch.tensor([n_pairs], device="cuda", dtype=torch.int64); dist.all_reduce(tp); total_pairs = int(tp.item())
    value = total_pairs * args.steps / (ms / 1e3)
    tiles = eng.tile_counts()

    e2e_growth = args.growth
    hparts, h2d_bytes = stage_e2e_shards(e2e_growth)
    for _ in range(max(args.warmup, 3)):
        step_e2e()
    gather_flush()
    # the staging producer adapts its shard schedule to the measured copy / kernel ratio of this rank (several ranks
    # share the host's PCIe paths, so the copies are slower at N > 1): shard k+1 may be kernel_ms / h2d_ms times larger
    # than shard k and still hide its copy
    if args.growth > 1.0:
        tw = eng.timing()
        g_new = pick_growth(tw["h2d_ms"], tw["prep_ms"] + tw["sw_ms"] + tw["post_ms"], args.growth)
        if world > 1:      # every rank must take the same branch (the extra warm-up steps below contain a collective)
            tg = torch.tensor([g_new], device="cuda", dtype=torch.float64); dist.all_reduce(tg, op=dist.ReduceOp.MIN); g_new = float(tg.item())
        if abs(g_new - e2e_growth) > 0.05:
            e2e_growth = g_new
            hparts, h2d_bytes = stage_e2e_shards(e2e_growth)
            for _ in range(2):
                step_e2e()
            gather_flush()
    ms_e, _, _, last_e, _ = timed(step_e2e, args.steps)
    t_e = eng.timing()
    e2e_value = total_pairs * args.steps / (ms_e / 1e3)
    n_local = len(last_e.row)
    n_out = n_local
    if world > 1:
        tn = torch.tensor([n_out], device="cuda", dtype=torch.int64); dist.all_reduce(tn); n_out = int(tn.item())
    d2h_bytes = n_out * 16 + 32 * world    # row, col (u32) + val (f64) per triplet (VTX_F_VALUES_ONLY) + counters, all ranks
    if world > 1:
        tb = torch.tensor([h2d_bytes], device="cuda", dtype=torch.int64); dist.all_reduce(tb); h2d_total = int(tb.item())
    else:
        h2d_total = h2d_bytes

    # gather_check (N > 1): one more step outside the timed region; the gathered matrix must hold exactly the ranks' triplets
    gather_check = None
    if world > 1:
        loc = step_e2e()
        local_sum = triplet_checksum(loc.row, loc.col, loc.val)
        n_loc = len(loc.row)
        gres = gather_flush()
        agg = torch.tensor([n_loc, local_sum & 0x7FFFFFFFFFFFFFFF, local_sum >> 63], device="cuda", dtype=torch.int64)
        parts = [torch.zeros_like(agg) for _ in range(world)]
        dist.all_gather(parts, agg)
        if rank == 0 or args.gather == "all":
            full = eng.fetch(gres, copy=False)
            want_n = sum(int(p[0]) for p in parts)
            want_sum = sum((int(p[2]) << 63) | int(p[1]) for p in parts) & 0xFFFFFFFFFFFFFFFF
            key = full.row.astype(np.int64) * (1 << 32) + full.col
            gather_check = bool(int(gres.n) == want_n == len(full.row) and triplet_checksum(full.row, full.col, full.val) == want_sum
                                and (len(key) < 2 or bool((np.diff(key) > 0).all())))

    line = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0)); peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6.65 TB/s"
        b_alg = vb.synth.algorithmic_bytes_per_pair(info)
        traffic, traffic_src, alu_pct, tj_kernel = None, None, None, "vtx_k_sw_fold"
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "sw_kernel_traffic.json")))
            traffic = tj["dram_bytes_per_pair"] * n_pairs; traffic_src = tj["source"]; alu_pct = tj.get("alu_pipe_active_pct")
            tj_kernel = tj.get("kernel", tj_kernel)
        except Exception:
            pass
        sw_avg_ms = float(np.mean(sw_ms))
        achieved = n_pairs * b_alg / (sw_avg_ms / 1e3) / 1e9
        cells = info["read_len"] * 2 * (2 * 100 + 1)
        # the bound that actually binds: the ALU pipe.  DPX s16x2 instructions (and PRMT) occupy it for 2 cycles per warp
        # and SMSP, 32-bit VIADD / IADD3 / LOP3 / SEL / ISETP for 1 (profiles/r01_dpx_microbench.txt).  Counted from the SASS
        # of the kernel that took the work (DESIGN.md section 4):
        #   folded kernel, tile = 4 pairs: main-pass warp-step (12 columns, forward | reverse halves) = 54 DPX + 19 -> 127
        #     cycles, (m + 7) steps; allele-column warp-step (19 rows) = 86 DPX + 28 -> 200 cycles, (L + 7) steps for L allele
        #     columns; boundary unpack 135; junction 199 (8 more, divergent, when the alleles differ in length)
        #   two-phase kernel, tile = 8 pairs: phase-1 warp-step 128 cycles x (m + 7), phase-2 warp-step (27 columns) 280 x (m + 3)
        m = info["read_len"]
        folded = tiles[7] * 4 >= sum(tiles[:4]) * 4 + sum(tiles[5:7]) * 8
        if folded:
            lmax = np.maximum(sb.ref_len, sb.alt_len).astype(np.float64) - 192.0
            uneq = float(np.mean(sb.ref_len != sb.alt_len))
            alu_cycles_per_pair = ((m + 7) * 127.0 + (float(lmax.mean()) + 7) * 200.0 + 135 + 199 + uneq * 8 * 199) / 4.0
            model_kernel = "folded SW kernel vtx_k_sw_fold"
        else:
            alu_cycles_per_pair = ((m + 7) * 128.0 + (m + 3) * 280.0) / 8.0
            model_kernel = "two-phase SW kernel vtx_k_sw_split<0>"
        sm_mhz = (clocks or {}).get("sm_mhz") or float(peaks.get("sm_max_mhz", 1965.0))
        dpx_peak = torch.cuda.get_device_properties(local).multi_processor_count * 4.0 * sm_mhz * 1e6
        dpx_ach = n_pairs * alu_cycles_per_pair / (sw_avg_ms / 1e3)
        extra = {"device_submits_per_step": len(dparts)}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "int16x2", "data": "synthetic", "config": describe(args, cfg, world, info, extra),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_total, "d2h_bytes_per_step": d2h_bytes,
                    "h2d_bytes_per_candidate": h2d_bytes / max(info["n_cand"], 1),
                    "shards_per_step": len(hparts), "shard_growth": e2e_growth,
                    "ms_per_step": ms_e / args.steps,
                    "last_step_device_ms": {k: round(t_e[k], 3) for k in ("h2d_ms", "prep_ms", "sw_ms", "post_ms")}},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "ncu_alu_pipe_active_pct": alu_pct,
                         "peak_source": peak_src, "kernel": tj_kernel,
                         "kernel_ms": sw_avg_ms, "algorithmic_bytes_per_pair": b_alg, "pairs_per_launch": n_pairs / max(len(dparts), 1),
                         "gcups": n_pairs * cells / (sw_avg_ms / 1e3) / 1e9,
                         "issue_bound": {"what": "ALU-pipe busy cycles/s of the %s (SASS model: %.0f SMSP-cycles per pair)" % (model_kernel, alu_cycles_per_pair),
                                         "tiles_per_kernel_class": tiles,
                                         "achieved": dpx_ach, "peak": dpx_peak, "frac": dpx_ach / dpx_peak,
                                         "peak_source": "n_SM x 4 SMSPs x sampled SM clock; DPX = 2 cycles, VIADD = 1 (measured, profiles/r01_dpx_microbench.txt)"},
                         "note": "integer DP: ~540 cell updates per algorithmic byte, so the kernel is DPX-issue bound, not HBM "
                                 "bound (DESIGN.md); gcups = DP cell updates/s of the SW kernel alone"},
            "clocks": clocks,
        }
        if gather_check is not None:
            line["gather_check"] = gather_check
        if not args.no_cpu_baseline:        # rank 0, also at N > 1 (the other ranks wait at the barrier below)
            os.sched_setaffinity(0, full_affinity)
            line["cpu_baseline"] = cpu_baseline(sb, bcs, cfg, info, args.cpu_seconds)
    eng.close()
    if world > 1:
        dist.barrier(); dist.destroy_process_group()
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    if line:
        print(json.dumps(line), flush=True)
    return 0


def main():
    args = parse_args()
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes what the CUDA path computed (--impl vartrix_b200)")
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
