#!/usr/bin/env python
"""Benchmark of the orgscorer hot path (contract: see the task statement / DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the whole hot path (K1..K10) over one batch of synthetic contigs of
BASELINE.json's configs[1] shape (cfg2: 100k contigs per GPU, 2-8 genes, ~50 hits/gene, 5k species).
`value`  : contigs/s, device-timed (CUDA events on the engine's stream), inputs resident in HBM (wide 29 B/hit layout,
           the per-unit figure of SURVEY 8d).
`e2e`    : same metric through the C-ABI plugin call with pinned HOST buffers (compact 14 B/hit wire format when the
           batch allows it): H2D + kernels + compaction + D2H of the results inside the timed region.
N > 1    : one process per GPU (torchrun).  ONE global batch (N tiles of the 100k-contig batch) is cut with
           waafle_b200.dist.shard_bounds; every rank scores its shard (weak scaling, no data-path collective), and
           every e2e step ends with the NCCL gather of the packed result records to rank 0 from device buffers on the
           engine's stream, followed by rank 0's D2H of the gathered whole.  Time = max over ranks; after the timed
           loop rank 0 checks the gathered whole against the C restatement of the reference.
`strong` : configs[2] (1M contigs total, 8-level taxonomy) cut over the N ranks the same way (strong scaling).
--impl reference : the UNMODIFIED reference (oracle/_ref, installed by oracle/build_ref.py) on all host cores, one
           process per core, on a bounded sample of the same workload; the numpy port if the install is missing.
--dump-outputs DIR : after the timed steps, the results of the last device-resident step (what `value` timed; rank 0's
           shard when N > 1) as DIR/<name>.npy in float64, at most 64 MB in all.  The workload is seeded, so two builds
           can be compared array for array.
"""

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "contigs/sec scored+classified"
UNIT = "contigs/s"
FALLBACK_HBM_GBS = 6650.0   # /opt/skills/guides/B200_PROFILING.md fallback
SCORE_RTOL = 1e-12          # north_star tolerance on emitted scores (calls / clades / loci are bit-exact)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2")
    ap.add_argument("--contigs", type=int, default=None, help="contigs per GPU (default: config size)")
    ap.add_argument("--cpu-sample", type=int, default=None, help="contigs in the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the configs[2] strong-scaling leg")
    ap.add_argument("--strong-contigs", type=int, default=1_000_000)
    ap.add_argument("--no-stream", action="store_true", help="skip the configs[4] streaming leg")
    ap.add_argument("--stream-contigs", type=int, default=10_000_000)
    ap.add_argument("--stream-chunk", type=int, default=125_000, help="contigs per streamed chunk")
    ap.add_argument("--exact", action="store_true", help="exact pipeline for every contig (bit-exact crit / rank)")
    ap.add_argument("--wide", action="store_true", help="e2e leg with the wide 29 B/hit wire format")
    ap.add_argument("--opt", action="append", default=[], help="engine option name=value (wfl_set_option)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's result arrays to DIR/<name>.npy (float64, <= 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the CUDA engine's results: it needs --impl ours")
    return args


DUMP_BYTES = 64 * 10 ** 6   # --dump-outputs: all .npy files together, headers included
NPY_HEADER = 128            # bytes np.save writes before the data of a 1-d or 2-d array


def dump_outputs(res, out_dir, limit=DUMP_BYTES):
    """Every non-empty result array as <out_dir>/<name>.npy in float64 (exact for the engine's integer outputs); an array
    without elements (ann_winner of a workload without annotation systems) carries no output and is not written.  When the
    whole would exceed `limit`, each array larger than a common byte budget keeps that many rows, chosen by a generator
    seeded with 0; arrays of the same length (the per-contig ones, the per-locus ones) therefore keep the same rows, and
    small arrays such as call_counts stay whole.  Returns the bytes written."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v) for k, v in res.items() if np.asarray(v).size > 0}
    room = limit - NPY_HEADER * len(arrays)
    sizes = sorted(8 * a.size for a in arrays.values())
    cap = room
    if sum(sizes) > room:   # largest per-array budget `cap` with sum(min(size, cap)) <= room
        left, n_big = room, len(sizes)
        for s in sizes:
            if s * n_big > left:
                break
            left, n_big = left - s, n_big - 1
        cap = left // n_big
    written = 0
    for name, a in arrays.items():
        if 8 * a.size > cap:
            keep = cap // (8 * (a.size // len(a)))
            a = a[np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))]
        path = os.path.join(out_dir, name + ".npy")
        np.save(path, a.astype(np.float64))
        written += os.path.getsize(path)
    return written


# --------------------------------------------------------------------------------------------
# CPU arms.  (1) the unmodified reference through oracle/reference_harness.py, one process per core, on text files
# of a sample of the workload; (2) the numpy port (oracle/orgscorer_oracle.py), same sharding; (3) the C restatement
# (oracle/orgscorer_oracle.c, one thread per core) on the whole workload: also the full-size parity reference.
# --------------------------------------------------------------------------------------------

def _oracle_worker(job):
    from oracle import orgscorer_oracle as oracle
    params, tax, arrays = job
    t = time.perf_counter()
    out = oracle.score_batch(params, tax, arrays)
    return time.perf_counter() - t, out["call_counts"].tolist()


def port_run(batch, params, tax, n_sample, cores):
    """Wall-clock contigs/s of the numpy port over `n_sample` contigs using `cores` processes."""
    import multiprocessing as mp
    n_sample = min(n_sample, batch.n_contigs)
    cores = max(1, min(cores, n_sample))
    cuts = np.linspace(0, n_sample, cores + 1).astype(int)
    jobs = [(params.as_dict(), tax.tables(), batch.slice(int(a), int(b)).arrays())
            for a, b in zip(cuts[:-1], cuts[1:]) if b > a]
    ctx = mp.get_context("fork")
    t0 = time.perf_counter()
    with ctx.Pool(len(jobs)) as pool:
        pool.map(_oracle_worker, jobs)
    wall = time.perf_counter() - t0
    return n_sample / wall, wall, len(jobs)


class ReferenceArm:
    """The unmodified waafle_orgscorer on `n_sample` contigs of a synthetic workload, one process per core."""

    def __init__(self, data, n_sample, cores):
        from oracle import reference_harness as rh
        self.rh = rh
        self.n_sample = min(n_sample, data.n_contigs)
        self.cores = max(1, min(cores, self.n_sample))
        self.dir = tempfile.mkdtemp(prefix="wfl_ref_")
        cuts = np.linspace(0, self.n_sample, self.cores + 1).astype(int)
        self.files = [data.write_files(self.dir, "shard{}".format(k), int(a), int(b))
                      for k, (a, b) in enumerate(zip(cuts[:-1], cuts[1:])) if b > a]

    @staticmethod
    def available():
        from oracle import reference_harness as rh
        return rh.available()

    def step(self):
        """(wall seconds incl. the reference's parsers, engine-only seconds = slowest process inside OS:952-960)."""
        wall, engine, total, calls = self.rh.time_reference_sharded(self.files)
        return wall, engine

    def close(self):
        import shutil
        shutil.rmtree(self.dir, ignore_errors=True)


def make_workload(args, workload=None, contigs=None):
    from waafle_b200 import synth
    from waafle_b200.params import OrgscorerParams
    data = synth.generate_config(workload or args.workload, n_contigs=contigs or args.contigs, seed=1000)
    tax = data.taxonomy()
    batch = data.to_batch(tax).sort_hits()   # what the front end's packer delivers (packing.pack)
    params = OrgscorerParams(n_systems=1 if batch.hit_sysmask is not None else 0)
    return data, batch, params, tax


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True,
                                     timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


def workload_name(workload, n):
    desc = {"cfg2": "synthetic {} contigs, 2-8 genes, ~50 hits/gene, 5k-species taxonomy (BASELINE configs[1])",
            "cfg3": "synthetic {} contigs, 2-20 genes, 8-level taxonomy (BASELINE configs[2] shape)",
            "cfg4": "long-contig stress {} contigs, 100-130 genes, 550-species pools (BASELINE configs[3] shape)",
            "cfg5": "Prodigal-style {} contigs, short/empty loci, annotations (BASELINE configs[4] shape)"}
    return desc[workload].format(n)


def run_reference(args, rank, world):
    """CPU arm: rank 0 alone times the reference's own CPU implementation on a bounded sample of the workload."""
    if rank != 0:
        return
    from waafle_b200 import synth
    cores = os.cpu_count() or 1
    n_cfg = args.contigs or synth.CONFIGS[args.workload]["n_contigs"]
    if ReferenceArm.available():
        per_core = {"cfg2": 100, "cfg3": 40, "cfg5": 40, "cfg4": 1}.get(args.workload, 40)
        n_sample = args.cpu_sample or cores * per_core
        data = synth.generate_config(args.workload, n_contigs=max(n_sample, 64), seed=1000)
        arm = ReferenceArm(data, n_sample, cores)
        walls, engines = [], []
        for step in range(args.warmup + args.steps):
            w, e = arm.step()
            if step >= args.warmup:
                walls.append(w)
                engines.append(e)
        arm.close()
        used, kind = arm.cores, "reference"
        n_sample = arm.n_sample
        # the path is the engine region waafle_orgscorer.py:952-960: the value is timed INSIDE it (slowest process), so
        # that the reference's text parsing -- which the GPU arm's packed host buffers do not pay either -- stays out
        T = sum(engines)
        sample = ("{} contigs of {} per step as blastout / GFF / taxonomy text files, UNMODIFIED waafle_orgscorer "
                  "(oracle/_ref, driven by oracle/reference_harness.py), one process per core; value = time inside the "
                  "engine region waafle_orgscorer.py:952-960 (slowest process)".format(n_sample, args.workload))
        extra = {"with_parsers": {"value": n_sample * args.steps / sum(walls), "unit": UNIT,
                                  "what": "same runs, wall clock incl. the reference's parsers and process start-up"}}
    else:
        per_core = {"cfg2": 400, "cfg3": 150, "cfg5": 150, "cfg4": 2}.get(args.workload, 100)
        n_sample = args.cpu_sample or cores * per_core
        a2 = argparse.Namespace(**vars(args))
        data, batch, params, tax = make_workload(a2, contigs=max(n_sample, 64))
        times = []
        for step in range(args.warmup + args.steps):
            rate, wall, used = port_run(batch, params, tax, n_sample, cores)
            if step >= args.warmup:
                times.append(wall)
        T, kind, extra = sum(times), "port", {}
        sample = ("{} contigs of {} per step, numpy oracle (restatement of the reference's Python/numpy orgscorer; "
                  "oracle/_ref not installed), one process per core".format(n_sample, args.workload))
    value = n_sample * args.steps / T
    cb = {"value": value, "unit": UNIT, "cores": used, "kind": kind, "sample": sample}
    cb.update(extra)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * T / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": workload_name(args.workload, n_cfg), "sample_contigs_per_step": n_sample},
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def cpu_baseline_leg(args, data, batch, params, tax):
    """N=1 only: the reference (or its port) on a bounded sample, and the C restatement on the whole workload."""
    cores = os.cpu_count() or 1
    if ReferenceArm.available():
        per_core = {"cfg2": 250, "cfg3": 100, "cfg5": 100, "cfg4": 1}.get(args.workload, 60)
        arm = ReferenceArm(data, args.cpu_sample or cores * per_core, cores)
        wall, engine = arm.step()
        arm.close()
        cb = {"value": arm.n_sample / engine, "unit": UNIT, "cores": arm.cores, "kind": "reference",
              "sample": "first {} contigs of the workload as text files, UNMODIFIED waafle_orgscorer (oracle/_ref), {} "
                        "processes; value = time inside the engine region waafle_orgscorer.py:952-960 (slowest process, "
                        "{:.1f} s)".format(arm.n_sample, arm.cores, engine),
              "with_parsers": {"value": arm.n_sample / wall, "unit": UNIT,
                               "what": "wall clock incl. the reference's parsers and process start-up ({:.1f} s)".format(wall)}}
    else:
        per_core = {"cfg2": 1500, "cfg3": 600, "cfg5": 600, "cfg4": 4}.get(args.workload, 300)
        n_sample = args.cpu_sample or cores * per_core
        rate, wall, used = port_run(batch, params, tax, n_sample, cores)
        cb = {"value": rate, "unit": UNIT, "cores": used, "kind": "port",
              "sample": "first {} contigs of the workload, numpy oracle, {} processes, {:.1f} s wall"
                        .format(min(n_sample, batch.n_contigs), used, wall)}
    c_ref = None
    try:
        from oracle import c_oracle
        tc = time.perf_counter()
        c_ref = c_oracle.score_batch(params, tax, batch, threads=cores)
        wall_c = time.perf_counter() - tc
        cb["c_port"] = {"value": batch.n_contigs / wall_c, "unit": UNIT, "cores": cores,
                        "sample": "all {} contigs, C restatement of the reference, {} threads, {:.1f} s wall"
                                  .format(batch.n_contigs, cores, wall_c)}
    except Exception as exc:   # the checker failing to build must not hide the GPU numbers
        cb["c_port"] = {"unavailable": repr(exc)[:200]}
    return cb, c_ref


def parity_report(ref, got, n, rtol, against):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import compare_results
    diffs = compare_results(ref, got, score_rtol=rtol)
    return {"checked_contigs": int(n), "against": against, "bit_exact": not diffs, "score_rtol": rtol,
            "what": "calls, clades, synteny, locus flags, melded members, annotation winners bit-exact; crit / rank "
                    "within score_rtol (0 = bit-exact)",
            "diffs": [str(d)[:160] for d in diffs[:3]]}


class E2E:
    """The timed end-to-end step: plugin call on pinned host buffers and -- with N > 1 -- the NCCL gather of the packed
    result records to rank 0 from device buffers on the engine's stream, then rank 0's D2H of the gathered whole."""

    def __init__(self, eng, shard, params, tax, dist, wide):
        import torch
        from waafle_b200.engine import PinnedArena
        self.eng, self.dist, self.torch = eng, dist, torch
        self.pin = PinnedArena()
        self.packed = (not wide) and shard.can_pack(len(tax.tables()["parent"]), params.n_systems)
        wire = shard.to_packed(params.min_scov) if self.packed else shard.arrays()
        self.harr = {k: self.pin.like(np.ascontiguousarray(v)) for k, v in wire.items()}
        self.h2d_bytes = int(sum(v.nbytes for v in self.harr.values()))
        self.d2h_bytes = 0
        self.out = None
        self.host_buf = None
        self.sizes = None
        self.gather_ms = 0.0
        if dist is None:
            eng.use_pinned_results(True)

    def step(self):
        torch = self.torch
        if self.dist is None:
            self.out = self.eng.score_batch(self.harr)
            self.d2h_bytes = int(sum(np.asarray(v).nbytes for v in self.out.values()))
            return
        from waafle_b200 import dist as wdist
        self.eng.score_batch_device(self.harr)
        blob, stream = wdist.device_blob(self.eng)
        with torch.cuda.stream(stream):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            gathered, sizes = wdist.gather_blobs(blob, self.dist)
            if gathered is not None:
                if self.host_buf is None or self.host_buf.shape != gathered.shape:
                    self.host_buf = torch.empty(gathered.shape, dtype=torch.uint8, pin_memory=True)
                self.host_buf.copy_(gathered, non_blocking=True)
                self.d2h_bytes = int(gathered.numel())
            e1.record(stream)
            stream.synchronize()
            self.gather_ms = e0.elapsed_time(e1)
        self.sizes = sizes

    def h2d_ceiling(self, barrier, reps=3):
        """Pure host->device copies of this rank's pinned wire buffers, all ranks at once: the bandwidth the box gives the
        plugin call's H2D window (ms per step's bytes, max over ranks is taken by the caller)."""
        torch = self.torch
        dst = {k: torch.empty(v.nbytes, dtype=torch.uint8, device="cuda") for k, v in self.harr.items()}
        src = {k: torch.from_numpy(v.view(np.uint8).reshape(-1)) for k, v in self.harr.items()}
        best = None
        for _ in range(reps):
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for k in dst:
                dst[k].copy_(src[k], non_blocking=True)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            best = ms if best is None else min(best, ms)
        return best

    def gathered_results(self, hit_bases):
        """rank 0, N > 1: the whole batch's results from the last step's gathered buffers."""
        from waafle_b200 import dist as wdist
        g = self.host_buf.numpy()
        return wdist.merge_blobs([g[r, :self.sizes[r]] for r in range(len(self.sizes))], hit_bases)

    def close(self):
        # the pinned staging tensor was used on the engine's stream: hand it back to torch's host allocator while that
        # stream still exists (the allocator records an event on it)
        self.host_buf = None
        if self.dist is not None:
            self.torch.cuda.synchronize()
        self.eng.use_pinned_results(False)
        self.pin.close()


def timed_e2e(e2e, steps, warmup, barrier):
    for _ in range(max(1, warmup)):
        e2e.step()
    barrier()
    t = time.perf_counter()
    for _ in range(steps):
        e2e.step()
    barrier()
    return 1e3 * (time.perf_counter() - t)


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    from waafle_b200 import dist as wdist
    from waafle_b200.packing import tiled_slice
    cores = wdist.bind_rank_to_cores(local_rank, int(os.environ.get("LOCAL_WORLD_SIZE", world))) if world > 1 else []

    # ---- the workload: ONE global batch = `world` tiles of the config's batch, cut by hit count ----
    data, base, params, tax = make_workload(args)
    n_base = base.n_contigs
    tile_hit_off = np.concatenate([[0]] + [base.hit_off[1:] + t * base.n_hits for t in range(world)])
    bounds = wdist.shard_bounds(tile_hit_off, world)
    c0, c1 = int(bounds[rank]), int(bounds[rank + 1])
    shard = base if world == 1 else tiled_slice(base, c0, c1)
    hit_bases = [int(tile_hit_off[b]) for b in bounds[:-1]]

    # ---- CPU baseline beside the GPU numbers (rank 0, N=1 only, before any CUDA init) ----
    cpu_baseline, c_ref = None, None
    if world == 1 and not args.no_cpu_baseline:
        cpu_baseline, c_ref = cpu_baseline_leg(args, data, base, params, tax)
    elif rank == 0 and not args.no_cpu_baseline:
        try:   # N > 1: only the C restatement, as the parity reference of the gathered whole
            from oracle import c_oracle
            c_ref = c_oracle.score_batch(params, tax, base, threads=max(1, len(cores)) if cores else (os.cpu_count() or 1))
        except Exception:
            c_ref = None

    import torch
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from waafle_b200.engine import Engine
    eng = Engine(local_rank, params, tax)
    if args.exact:
        eng.set_option("exact", 1)
    for kv in args.opt:
        k, v = kv.split("=")
        eng.set_option(k, int(v))
    rtol = 0.0 if args.exact else SCORE_RTOL

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident leg ("value") ----
    eng.upload(shard)
    for _ in range(args.warmup):
        eng.run_resident()
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    dev_ms, score_ms, launches = 0.0, 0.0, 0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        eng.run_resident()
        st = eng.stats()
        dev_ms += st["ms_kernels"]
        score_ms += st["ms_score_kernel"]
        launches += st["kernel_launches"]
    barrier()
    wall_ms = 1e3 * (time.perf_counter() - t0)
    res = eng.download()
    st = eng.stats()
    parity = None
    if world == 1 and c_ref is not None:
        parity = parity_report(c_ref, res, shard.n_contigs, rtol, "oracle/orgscorer_oracle.c")

    # ---- end-to-end leg: pinned host buffers through the plugin call (+ NCCL gather of the records for N > 1) ----
    e2e = E2E(eng, shard, params, tax, dist, args.wide)
    e2e_ms = timed_e2e(e2e, args.steps, args.warmup, barrier)
    st_e2e = eng.stats()
    gather_ms = e2e.gather_ms
    ceil_ms = e2e.h2d_ceiling(barrier)
    sampler.stop_flag = True
    sampler.join(timeout=2)
    if world > 1 and rank == 0:
        whole = e2e.gathered_results(hit_bases)
        if c_ref is not None:
            want = wdist.merge_results([c_ref] * world, [t * base.n_hits for t in range(world)])
            parity = parity_report(want, whole, n_base * world, rtol,
                                   "oracle/orgscorer_oracle.c (whole batch gathered to rank 0 over NCCL)")
    h2d_bytes, d2h_bytes = e2e.h2d_bytes, e2e.d2h_bytes
    wire_format = "packed 14 B/hit" if e2e.packed else "wide 29 B/hit"
    e2e.close()

    # ---- strong scaling: configs[2] (1M contigs, 8 levels) cut over the ranks, same e2e step ----
    strong = None
    if not args.no_strong and args.workload == "cfg2":
        strong = strong_leg(args, eng, dist, world, rank, barrier, rtol)

    # ---- max over ranks ----
    stream = None
    if not args.no_stream and args.workload == "cfg2":
        stream = stream_leg(args, eng, dist, world, rank, barrier)

    tv = torch.tensor([dev_ms, score_ms, e2e_ms, wall_ms, gather_ms, ceil_ms], dtype=torch.float64, device="cuda")
    hv = torch.tensor([float(h2d_bytes)], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(tv, op=dist.ReduceOp.MAX)
        dist.all_reduce(hv, op=dist.ReduceOp.SUM)
    dev_ms, score_ms, e2e_ms, wall_ms, gather_ms, ceil_ms = tv.tolist()
    h2d_total = hv.item()
    n_total = n_base * world

    if rank == 0:
        # roofline of the scoring kernel(s): algorithmic bytes per step = 29 B/hit + 9 B/locus + 16 B/contig in,
        # 40 B/contig + G(1+4S) B out (SURVEY 8d), plus 29 B/hit again for every extra taxonomy level a contig is
        # evaluated at.
        H = np.diff(shard.hit_off)
        extra_levels = np.maximum(res["lifts"] - params.jump_taxonomy, 0)
        alg_bytes = shard.algorithmic_bytes(params.n_systems) + 29 * int((H * extra_levels).sum())
        peak, peak_src = FALLBACK_HBM_GBS, "fallback"
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
                peak, peak_src = float(json.load(fh)["hbm_gbs"]), "measured"
        except Exception:
            pass
        achieved = alg_bytes / (score_ms / args.steps * 1e-3) / 1e9
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as fh:
                tj = json.load(fh)
                if tj.get("workload") == args.workload and tj.get("contigs") == shard.n_contigs and \
                        tj.get("mode") == ("exact" if args.exact else "fast"):
                    traffic = tj["dram_bytes_per_launch"]
        except Exception:
            pass
        kernel_name = ("wfl_pipe_* (exact pipeline: prepare, then regroup / K2 sort / k2 / masks / one / two / lift per "
                       "taxonomy level)" if args.exact else
                       "wfl_fast_contigs (fused shared-memory kernel: match, gene scores, masks, one- / two-clade search "
                       "and lifts for all levels in one launch; + the exact pipeline for the contigs it hands back)")
        line = {
            "metric": METRIC, "value": n_total * args.steps / (dev_ms * 1e-3), "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(args.workload, n_base), "contigs_per_gpu": shard.n_contigs,
                       "hits_per_gpu": shard.n_hits, "loci_per_gpu": shard.n_loci,
                       "global_batch": "{} tile(s) of the {}-contig batch, cut by waafle_b200.dist.shard_bounds".format(world, n_base),
                       "flags": "reference defaults (k1=0.5 k2=0.8 meld/meld range=0.05 weak-loci=ignore)",
                       "mode": "exact" if args.exact else "fast path + guard bands (exact pipeline for fallbacks)",
                       "parallelism": "contig-sharded x{}".format(world),
                       "l2": "inputs ({:.0f} MB/GPU) exceed the 126 MB L2; no flush needed".format(
                           shard.algorithmic_bytes(params.n_systems) / 1e6),
                       "mean_levels_per_contig": float(st["levels"]) / max(1, shard.n_contigs),
                       "wall_ms_per_step": wall_ms / args.steps,
                       "cores_bound": len(cores) if cores else None},
            "e2e": {"value": n_total * args.steps / (e2e_ms * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": int(h2d_total), "d2h_bytes_per_step": d2h_bytes,
                    "ms_per_step": e2e_ms / args.steps, "wire_format": wire_format,
                    "h2d_aggregate_gbs": h2d_total / max(st_e2e["ms_h2d"], 1e-6) / 1e6,
                    "h2d_ceiling": {"ms_per_step_bytes": ceil_ms, "aggregate_gbs": h2d_total / max(ceil_ms, 1e-6) / 1e6,
                                    "what": "the same pinned buffers copied host->device by all ranks at once with nothing else "
                                            "running (best of 3, max over ranks): what this box's host side can feed"},
                    "results": "host arrays through wfl_score_batch" if world == 1 else
                               "packed records gathered to rank 0 over NCCL from device buffers, then D2H",
                    "nccl_gather_ms": gather_ms if world > 1 else None,
                    "last_call_ms": {"h2d_window": st_e2e["ms_h2d"], "kernels_window": st_e2e["ms_kernels"],
                                     "d2h": st_e2e["ms_d2h"], "host_syncs": st_e2e["host_syncs"]}},
            "gpu_launches": int(launches),
            "roofline": {"kernel": kernel_name, "bound": "hbm", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": int(alg_bytes),
                         "kernel_ms": score_ms / args.steps},
            "cpu_baseline": cpu_baseline,
            "parity": parity,
            "strong": strong,
            "stream": stream,
            "clocks": sampler.summary(),
            "calls": {"lgt": int(res["call_counts"][0]), "no_lgt": int(res["call_counts"][1]),
                      "unclassified": int(res["call_counts"][2])},
            "engine_stats": {k: st[k] for k in ("matched_pairs", "groups", "levels", "pairs_tested",
                                                "pairs_scored", "workspace_retries", "smem_contigs", "fallback_contigs",
                                                "guard_trips", "refined_groups", "host_syncs")},
        }
        print(json.dumps(line))
    if args.dump_outputs and rank == 0:   # `res`: plain host arrays of the last resident step, untouched by the later legs
        nbytes = dump_outputs(res, args.dump_outputs)
        print("dumped {:.1f} MB of results to {}".format(nbytes / 1e6, args.dump_outputs), file=sys.stderr)
    eng.close()
    if dist is not None:
        dist.destroy_process_group()


def strong_leg(args, eng, dist, world, rank, barrier, rtol):
    """configs[2]: `--strong-contigs` contigs in total (8 tiles of a generated eighth), full 8-level taxonomy, default
    flags, cut over the ranks by hit count; e2e step incl. the gather; parity of the gathered whole on rank 0."""
    import torch
    from waafle_b200 import dist as wdist
    from waafle_b200.packing import tiled_slice
    total = args.strong_contigs
    tiles = 8
    a3 = argparse.Namespace(**vars(args))
    data3, base3, params3, tax3 = make_workload(a3, workload="cfg3", contigs=max(1, total // tiles))
    n3 = base3.n_contigs
    tile_off = np.concatenate([[0]] + [base3.hit_off[1:] + t * base3.n_hits for t in range(tiles)])
    bounds = wdist.shard_bounds(tile_off, world)
    c0, c1 = int(bounds[rank]), int(bounds[rank + 1])
    shard3 = tiled_slice(base3, c0, c1)
    hit_bases = [int(tile_off[b]) for b in bounds[:-1]]
    ref3 = None
    if rank == 0 and not args.no_cpu_baseline:
        try:
            from oracle import c_oracle
            ref3 = c_oracle.score_batch(params3, tax3, base3, threads=os.cpu_count() or 1)
        except Exception:
            ref3 = None
    eng.set_params(params3)
    eng.set_taxonomy(tax3)
    e2e = E2E(eng, shard3, params3, tax3, dist, args.wide)
    steps = args.steps
    ms = timed_e2e(e2e, steps, 1, barrier)
    st = eng.stats()
    parity = None
    if rank == 0 and ref3 is not None:
        whole = e2e.gathered_results(hit_bases) if dist is not None else e2e.out
        want = wdist.merge_results([ref3] * tiles, [t * base3.n_hits for t in range(tiles)])
        parity = parity_report(want, whole, n3 * tiles, rtol, "oracle/orgscorer_oracle.c")
    tv = torch.tensor([ms, st["ms_kernels"], e2e.gather_ms], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(tv, op=dist.ReduceOp.MAX)
    ms, k_ms, g_ms = tv.tolist()
    out = {"workload": workload_name("cfg3", n3 * tiles) + ": {} tiles of a generated {}-contig batch".format(tiles, n3),
           "scaling": "strong", "contigs_total": n3 * tiles, "hits_total": int(base3.n_hits) * tiles,
           "value": n3 * tiles * steps / (ms * 1e-3), "unit": UNIT, "steps": steps, "ms_per_step": ms / steps,
           "what": "e2e: pinned host buffers -> plugin call -> (N > 1: NCCL gather of the packed records to rank 0) -> D2H",
           "kernels_window_ms": k_ms, "nccl_gather_ms": g_ms if dist is not None else None,
           "wire_format": "packed 14 B/hit" if e2e.packed else "wide 29 B/hit", "parity": parity,
           "engine_stats": {k: st[k] for k in ("levels", "smem_contigs", "fallback_contigs", "guard_trips",
                                               "refined_groups", "workspace_retries")}}
    e2e.close()
    return out


def stream_leg(args, eng, dist, world, rank, barrier):
    """configs[4]: `--stream-contigs` Prodigal-style contigs with annotation transfer under --weak-loci assign-unknown,
    streamed in chunks of `--stream-chunk` contigs; chunk k goes to rank k % N.  Every chunk is a full plugin call from
    pinned host buffers (H2D + kernels + compaction), its packed result records are read back to the host (what a writer
    would consume), and the call counts of all chunks are summed over the ranks at the end.  The chunks are tiles of one
    generated chunk (a 10M-contig synthetic set does not fit a build-time budget); rank 0 checks the chunk against the C
    restatement under all three --weak-loci modes."""
    import torch
    from waafle_b200 import dist as wdist
    from waafle_b200.engine import PinnedArena
    from waafle_b200.params import WEAK_LOCI, OrgscorerParams
    from waafle_b200 import synth
    data = synth.generate_config("cfg5", n_contigs=args.stream_chunk, seed=1000, annotations=True)
    tax5 = data.taxonomy()
    chunk = data.to_batch(tax5).sort_hits()
    n_chunks = max(1, (args.stream_contigs + chunk.n_contigs - 1) // chunk.n_contigs)
    mine = len(range(rank, n_chunks, world))
    modes = ("assign-unknown", "penalize", "ignore")
    eng.set_taxonomy(tax5)
    parity = None
    if rank == 0 and not args.no_cpu_baseline:
        from oracle import c_oracle
        parity = {}
        for mode in modes:
            P = OrgscorerParams(n_systems=1, weak_loci=WEAK_LOCI[mode])
            eng.set_params(P)
            ref = c_oracle.score_batch(P, tax5, chunk, threads=os.cpu_count() or 1)
            parity[mode] = parity_report(ref, eng.score_batch(chunk), chunk.n_contigs, SCORE_RTOL,
                                         "oracle/orgscorer_oracle.c")["bit_exact"]
    P = OrgscorerParams(n_systems=1, weak_loci=WEAK_LOCI[modes[0]])
    eng.set_params(P)
    pin = PinnedArena()
    packed = chunk.can_pack(len(tax5.tables()["parent"]), 1)
    wire = chunk.to_packed(P.min_scov) if packed else chunk.arrays()
    harr = {k: pin.like(np.ascontiguousarray(v)) for k, v in wire.items()}
    h2d = int(sum(v.nbytes for v in harr.values()))
    host_buf, counts, d2h = None, np.zeros(3, np.int64), 0

    def one_chunk():
        nonlocal host_buf, d2h
        eng.score_batch_device(harr)
        blob, stream = wdist.device_blob(eng)
        with torch.cuda.stream(stream):
            if host_buf is None or host_buf.numel() < blob.numel():
                host_buf = torch.empty(blob.numel(), dtype=torch.uint8, pin_memory=True)
            host_buf[:blob.numel()].copy_(blob, non_blocking=True)
            stream.synchronize()
        d2h = int(blob.numel())
        return blob.numel()

    nb = one_chunk()   # warm-up (allocations)
    from waafle_b200.engine import unpack_results
    one = unpack_results(host_buf.numpy()[:nb])["call_counts"]
    barrier()
    t = time.perf_counter()
    kms = 0.0
    for _ in range(mine):
        one_chunk()
        counts += one
        kms += eng.stats()["ms_kernels"]
    barrier()
    ms = 1e3 * (time.perf_counter() - t)
    tv = torch.tensor([ms, kms], dtype=torch.float64, device="cuda")
    cv = torch.tensor(counts.tolist() + [mine], dtype=torch.int64, device="cuda")
    if dist is not None:
        dist.all_reduce(tv, op=dist.ReduceOp.MAX)
        dist.all_reduce(cv, op=dist.ReduceOp.SUM)
    ms, kms = tv.tolist()
    tot = cv.tolist()
    host_buf = None
    torch.cuda.synchronize()
    pin.close()
    n_total = tot[3] * chunk.n_contigs
    return {"workload": workload_name("cfg5", n_total) + ": {} chunks of {} contigs, chunk k on rank k % {}".format(
                tot[3], chunk.n_contigs, world),
            "flags": "--weak-loci assign-unknown, annotation transfer (1 system)", "contigs_total": n_total,
            "hits_total": int(chunk.n_hits) * tot[3], "value": n_total / (ms * 1e-3), "unit": UNIT,
            "seconds": ms * 1e-3, "kernels_ms_max_rank": kms,
            "what": "per chunk: pinned host buffers -> plugin call -> packed result records D2H; counts all-reduced at the end",
            "h2d_bytes_per_chunk": h2d, "d2h_bytes_per_chunk": d2h,
            "wire_format": "packed 15 B/hit" if packed else "wide 33 B/hit",
            "calls": {"lgt": tot[0], "no_lgt": tot[1], "unclassified": tot[2]},
            "parity_one_chunk_vs_c_oracle": parity}


if __name__ == "__main__":
    main()
