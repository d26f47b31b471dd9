#!/usr/bin/env python
"""bench.py -- queries/sec of the raxtax query-classification hot path on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W                   our CUDA path (one process per GPU under torchrun)
  python bench.py --impl reference --gpus N --steps K --warmup W  the reference algorithm on the host cores (CPU oracle port)

A "step" is one pass of the hot path (k-mers -> hit counts -> probabilities -> lineage results) over the workload's queries.

Workloads (--workload, BASELINE.json configs):
  c3 (default)  1 M COI-like 650 bp references x 200 k queries IN TOTAL, index replicated, the queries split evenly over the N
                ranks (strong scaling, no data-path collective) -- the configuration the metric's 1/2/4/8 series is quoted on
  c2            100 k references x 10 k queries per GPU (the single-GPU config; weak scaling when N > 1)
  c4            500 k 16S-like 1500 bp references x 100 k queries in total, --skip-exact-matches (strong scaling)
  c5            8 M references sharded over the N ranks, every rank sees every query, NCCL histogram all-reduce + record
                all-gather inside the device library (bounded query job, see --queries)

Legs of one run, all over the same queries:
  value            whole-job queries/s with the batch resident in HBM (rtx_batch_run, CUDA events on the context's stream)
  e2e              the same through the drop-in driver rxh_raxtax (raxtax.rs:14-97): host query arrays in, exact-match lookup,
                   de-duplication, H2D, kernels, D2H, formatting of every result line and the per-query hand-off to a counting
                   sender all inside the timed region (host wall clock, barrier on both sides, max over ranks)
  e2e_device_abi   rtx_classify_batch with page-locked host buffers (the device boundary alone: H2D + kernels + D2H)
  roofline         the hit-count kernel, from per-launch CUDA events with the kernels serialised
  cpu_baseline     the CPU oracle port on the host cores over a bounded sample (rank 0, N = 1 only)

--dump-outputs DIR writes the result arrays of the value leg's last timed step (c5: of its timed leg) as .npy files (dump_outputs): the
inputs are seeded, so two builds run with the same arguments can be compared output for output.
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

METRIC = "queries/sec (box, device-timed) at 1/2/4/8 B200; hit-count HBM GB/s vs peak"
UNIT = "queries/s"

# name -> (scaling, skip_exact_matches)
WORKLOADS = {"c2": ("weak", False), "c3": ("strong", False), "c4": ("strong", True), "c5": ("strong", False)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed regions: NVML polled every ~10 ms from a thread; falls back to an
    nvidia-smi loop when pynvml is missing."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []
        self.nvml = None
        self.samples = []  # (sm_mhz, reasons bitmask)
        self.stop_flag = False
        self.t = None
        try:
            import pynvml

            pynvml.nvmlInit()
            # NVML enumerates physical devices: honour CUDA_VISIBLE_DEVICES when it is a plain list of ordinals
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            idx = gpu_index
            if vis and all(x.strip().isdigit() for x in vis.split(",")):
                idx = int(vis.split(",")[gpu_index])
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                self.samples.append((float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)), int(n.nvmlDeviceGetCurrentClocksEventReasons(self.h))))
            except Exception:
                try:
                    self.samples.append((float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)), int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))))
                except Exception:
                    break
            time.sleep(0.01)

    def start(self):
        if self.nvml is not None:
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.gpu)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.t.join(timeout=1)
            n = self.nvml
            names = {"hw_slowdown": getattr(n, "nvmlClocksEventReasonHwSlowdown", 0x8), "hw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                     "sw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonSwThermalSlowdown", 0x20), "sw_power_cap": getattr(n, "nvmlClocksEventReasonSwPowerCap", 0x4)}
            sm = [x[0] for x in self.samples]
            reasons = sorted(k for k, bit in names.items() if any(x[1] & bit for x in self.samples))
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.smax, "reasons": reasons, "samples": len(sm), "source": "nvml, 10 ms poll"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower() == "active":
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(smax)) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 200"}


# ---------------------------------------------------------------------------------------------------------------------
def load_workload(name, n_queries, rank=0, barrier=None):
    """The synthetic data set of a BASELINE config (raxtax_b200/synth.py, deterministic).  Generating 1 M references takes ~40 s of
    numpy, so the arrays are cached under /tmp: the reference arm, our arm and the ranks of a multi-GPU run on one box then share
    one generation (rank 0 writes, the others wait at the barrier and read)."""
    from raxtax_b200 import synth

    path = os.path.join(os.environ.get("RAXTAX_BENCH_CACHE", "/tmp"), f"raxtax_b200_synth_{name}_{n_queries}_v2.npz")

    def from_cache():
        z = np.load(path, allow_pickle=False)
        return synth.Dataset(name, bytes(z["lin"]).decode().split("\n"), z["ref_off"], z["ref_codes"], bytes(z["qlab"]).decode().split("\n"),
                             z["q_off"], z["q_codes"], meta=json.loads(bytes(z["meta"]).decode()))

    ds = None
    if os.path.exists(path):
        try:
            ds = from_cache()
        except Exception:
            ds = None
    if ds is None and rank == 0:
        ds = synth.generate(name, n_queries=n_queries, measure=False)
        try:
            tmp = path + f".{os.getpid()}.tmp.npz"
            np.savez(tmp, lin=np.frombuffer("\n".join(ds.ref_lineages).encode(), np.uint8), ref_off=ds.ref_off, ref_codes=ds.ref_codes,
                     qlab=np.frombuffer("\n".join(ds.query_labels).encode(), np.uint8), q_off=ds.query_off, q_codes=ds.query_codes,
                     meta=np.frombuffer(json.dumps(ds.meta).encode(), np.uint8))
            os.replace(tmp, path)
        except Exception:
            pass
    if barrier is not None:
        barrier()
    if ds is None:
        try:
            ds = from_cache()
        except Exception:
            ds = synth.generate(name, n_queries=n_queries, measure=False)
    return ds


def workload_queries(name, world, override=0):
    """(queries in the whole job, queries per rank, scaling)"""
    from raxtax_b200 import synth

    scaling, _ = WORKLOADS[name]
    base = override or synth.CONFIGS[name][1]
    if name == "c5":
        return base, base, "strong"  # every rank sees every query; the references are what is split
    if scaling == "weak":
        return base * world, base, scaling
    per = (base + world - 1) // world
    return base, per, scaling


DUMP_BYTES = 60_000_000  # --dump-outputs: array bytes of one run, below 64 MB with the .npy headers
DUMP_SEED = 20261020


def dump_outputs(out, path, budget=DUMP_BYTES, first_query=0):
    """Writes one step's ClassifyOutput (what a caller of the timed path receives) as float32 / float64 .npy files under `path`, so
    that two builds can be compared output for output on the same inputs.  Every file is indexed by the queries in query.npy: all
    queries when everything fits in `budget` bytes, otherwise the longest prefix of a fixed seeded permutation of the queries that
    fits, in query order.  Per query: query (job-wide index), n_kmers, global_signal, n_results; per result line of those queries,
    in query order: first_ref, n_levels, confidence [lines, max levels] (zero past n_levels) and local_signal."""
    nq = len(out.n_kmers)
    rb = out.result_begin.astype(np.int64)
    n_lines = rb[1:] - rb[:-1]
    n_lev = out.confidence.shape[1]
    cost = (8 + 4 + 8 + 4) + n_lines * (8 + 4 + 8 * n_lev + 8)
    order = np.random.default_rng(DUMP_SEED).permutation(nq)
    q = np.sort(order[: int(np.searchsorted(np.cumsum(cost[order]), budget, side="right"))])
    cnt = n_lines[q]
    rows = np.repeat(rb[q] - (np.cumsum(cnt) - cnt), cnt) + np.arange(int(cnt.sum()))
    lev = out.n_levels[rows]
    conf = np.where(np.arange(n_lev)[None, :] < lev[:, None], out.confidence[rows], 0.0)
    os.makedirs(path, exist_ok=True)
    arrays = {"query": (q + first_query).astype(np.float64), "n_kmers": out.n_kmers[q].astype(np.float32),
              "global_signal": out.global_signal[q].astype(np.float64), "n_results": cnt.astype(np.float32),
              "first_ref": out.first_ref[rows].astype(np.float64), "n_levels": lev.astype(np.float32),
              "confidence": conf.astype(np.float64), "local_signal": out.local_signal[rows].astype(np.float64)}
    for k, a in arrays.items():
        np.save(os.path.join(path, f"{k}.npy"), a)
    print(f"--dump-outputs: {len(q)} of {nq} queries, {len(rows)} result lines -> {path}", file=sys.stderr)


class CpuReference:
    """The reference algorithm (oracle port of raxtax.rs:14-97 with the chunked thread fan-out of main.rs:119-124) on host cores,
    over a bounded sample of the workload's queries."""

    def __init__(self, ds, skip):
        from oracle import oracle as orc

        import ctypes as C

        self.orc = orc
        self.ds = ds
        self.skip = skip
        blob = "\n".join(ds.ref_lineages).encode()
        ro = np.ascontiguousarray(ds.ref_off, np.uint64)
        rc = np.ascontiguousarray(ds.ref_codes, np.uint8)
        t0 = time.time()
        self.tree = orc.Tree(orc.lib().orc_tree_new(ds.n_refs, blob, len(blob), ro.ctypes.data_as(C.POINTER(C.c_uint64)), rc.ctypes.data_as(C.POINTER(C.c_uint8))))
        self.tree_s = time.time() - t0

    def run(self, n, threads, chunk):
        ds = self.ds
        off = ds.query_off[: n + 1]
        o = self.tree.classify(off - off[0], ds.query_codes[int(off[0]): int(off[-1])], skip_exact=self.skip, threads=threads, chunk_size=chunk)
        return o["seconds"]

    def plan(self, q_total, threads, seconds_per_step, override=0):
        """(sample size, chunk): enough queries for ~seconds_per_step of work on all threads, every thread busy; chunks as the
        reference would cut them for the whole job (main.rs:119-124: max(100, Q / (threads * 10) + 1)) unless the sample is too small
        for that, in which case the sample is cut evenly (per-query cost does not depend on the chunk size)."""
        full_chunk = q_total if threads == 1 else max(100, q_total // (threads * 10) + 1)
        if override:
            n = min(q_total, override)
        else:
            probe = min(q_total, threads * 4)
            t = self.run(probe, threads, max(1, probe // threads))
            rate = probe / max(t, 1e-6)
            n = int(min(q_total, max(threads * 8, rate * seconds_per_step)))
            n = max(threads, n // threads * threads)
        chunk = full_chunk if n >= full_chunk * threads else max(1, n // threads)
        return n, chunk


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--queries", type=int, default=0, help="queries of the whole job (0 = the config's own number; c5 default: a bounded 131072)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="queries in the bounded CPU sample (0 = sized for ~20 s / ~6 s per step)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sharded", action="store_true", help="skip the reference-sharded check leg of a multi-GPU run")
    ap.add_argument("--sub-batch", type=int, default=0, help="RTX_OPT_SUB_BATCH for the timed legs (0 = library default)")
    ap.add_argument("--pipeline", type=int, default=-1, help="RTX_OPT_PIPELINE for the timed legs (-1 = library default)")
    ap.add_argument("--chunk", type=int, default=0, help="chunk_size of rxh_raxtax in the e2e leg (0 = the driver's default)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the timed leg returned in its last step to DIR/<name>.npy (see dump_outputs; DIR/rank<r>/ per rank when N > 1)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(min(args.warmup, 1), 1)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores = os.cpu_count() or 1
    # stdout carries the ONE JSON line and nothing else: whatever libraries print (NCCL writes its version banner to stdout) goes to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + "\n").encode())

    from raxtax_b200 import synth

    name = args.workload
    scaling, skip = WORKLOADS[name]
    if name == "c5" and not args.queries:
        args.queries = 131072
    ref_len, kind = synth.CONFIGS[name][2], synth.CONFIGS[name][3]
    kind_name = "16S-like" if kind == "16s" else "COI-like"

    # ------------------------------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        q_total, _, _ = workload_queries(name, max(args.gpus, 1), args.queries)
        ds = load_workload(name, q_total)
        ref = CpuReference(ds, skip)
        n_sample, chunk = ref.plan(q_total, cores, 6.0, args.cpu_sample)
        for _ in range(args.warmup):
            ref.run(n_sample, cores, chunk)
        secs = [ref.run(n_sample, cores, chunk) for _ in range(args.steps)]
        total = float(sum(secs))
        v = n_sample * args.steps / total
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "u16/f64",
                "data": "synthetic",
                "config": {"workload": f"{name}: {ds.n_refs} {kind_name} refs x {ref_len} bp (6-rank lineages) x {q_total} queries"
                                       + (", --skip-exact-matches" if skip else "") + f"; CPU arm: bounded sample of {n_sample} queries per step",
                           "oracle_tree_build_s": round(ref.tree_s, 1)},
                "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                 "sample": f"first {n_sample} queries of the {name} workload per step (chunks of {chunk}), {args.steps} steps, all {cores} host threads; "
                                           "C++ port of raxtax.rs / prob.rs / lineage.rs with flat count-indexed histogram tables (O(1) per reference like the "
                                           "reference's ahash maps); the Rust reference itself cannot be built in this image (no cargo / rustc)"},
                "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        emit(line)
        return 0

    # ------------------------------------------------------------------------------------------ our arm
    import torch
    import torch.distributed as dist

    from raxtax_b200 import capi

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    if name == "c5":
        from raxtax_b200 import bench_sharded

        line, out = bench_sharded.run(args, rank, local_rank, world, barrier, max_over_ranks, load_workload, ClockSampler, measured_peaks, METRIC, UNIT)
        if rank == 0:
            if args.dump_outputs:  # the lines of every query end up on rank 0
                dump_outputs(out, args.dump_outputs)
            emit(line)
        if world > 1:
            dist.destroy_process_group()
        return 0

    q_total, q_per_rank, scaling = workload_queries(name, world, args.queries)
    ds = load_workload(name, q_total, rank, barrier)
    t0 = time.time()
    tree = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes)
    t_tree = time.time() - t0
    ctx = capi.Context(local_rank)
    t0 = time.time()
    ctx.upload_tree(tree)
    t_upload = time.time() - t0
    q0 = min(rank * q_per_rank, q_total)
    q1 = min(q0 + q_per_rank, q_total)
    nq = q1 - q0
    off = (ds.query_off[q0: q1 + 1] - ds.query_off[q0]).astype(np.uint64)
    codes = ds.query_codes[int(ds.query_off[q0]): int(ds.query_off[q1])]
    eo, eids = tree.exact_batch(off, codes)
    # pinned host buffers for the device-ABI leg
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
    off_p, codes_p, eo_p, eids_p = pin(off), pin(codes), pin(eo), pin(eids if len(eids) else np.zeros(1, np.uint32))

    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local_rank))

    if args.sub_batch:
        ctx.set_option(capi.RTX_OPT_SUB_BATCH, args.sub_batch)
    if args.pipeline >= 0:
        ctx.set_option(capi.RTX_OPT_PIPELINE, args.pipeline)
    # ---- device-resident leg ------------------------------------------------------------------------------
    ctx.batch_upload(off_p, codes_p, eo_p, eids_p, skip_exact=skip)
    for _ in range(args.warmup):
        ctx.batch_run()
    ctx.synchronize()
    ctx.profile_reset()
    sampler = ClockSampler(local_rank)
    barrier()
    torch.cuda.synchronize()
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.steps):
        ctx.batch_run()
    ev1.record(stream)
    ctx.synchronize()
    torch.cuda.synchronize()
    barrier()
    dev_ms = max_over_ranks(ev0.elapsed_time(ev1))
    res = ctx.batch_download()
    prof_main = ctx.profile()
    n_results = len(res.first_ref)
    value = q_total * args.steps / (dev_ms / 1e3)
    sub_batch = ctx.sub_batch

    # ---- per-kernel leg: the same batch with every kernel timed by its own CUDA event pair on the launching stream (the
    # sub-batch pipeline off, so that every kernel runs alone on the GPU and its duration is its own)
    reps_k = max(1, min(args.steps, 3))
    ctx.set_option(capi.RTX_OPT_PIPELINE, 0)
    ctx.set_option(capi.RTX_OPT_SUB_BATCH, 0)
    ctx.set_option(capi.RTX_OPT_PROFILE, 1)
    ctx.batch_upload(off_p, codes_p, eo_p, eids_p, skip_exact=skip)
    ctx.batch_run()
    ctx.profile_reset()
    ser0, ser1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ser0.record(stream)
    for _ in range(reps_k):
        ctx.batch_run()
    ser1.record(stream)
    ctx.synchronize()
    serial_ms = ser0.elapsed_time(ser1) / reps_k
    ctx.batch_download()
    prof = ctx.profile()
    hit_kernel = ctx.hitcount_kernel_name()
    ctx.set_option(capi.RTX_OPT_PROFILE, 0)
    ctx.set_option(capi.RTX_OPT_PIPELINE, args.pipeline if args.pipeline >= 0 else 0)
    ctx.set_option(capi.RTX_OPT_SUB_BATCH, args.sub_batch)

    # ---- end-to-end leg: the drop-in driver (rxh_raxtax) over host query arrays, result strings into a counting sender ------
    queries = capi.Queries.new(ds.query_labels[q0:q1], off, codes)
    cnt = None
    for _ in range(2):
        cnt = capi.raxtax_counted(ctx, queries, tree, skip_exact_matches=skip, chunk_size=args.chunk)
    assert cnt["queries"] == nq, (cnt, nq)
    assert cnt["lines"] == n_results, f"the driver sent {cnt['lines']} result lines, the device-resident leg produced {n_results}"
    ctx.profile_reset()
    barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        c2 = capi.raxtax_counted(ctx, queries, tree, skip_exact_matches=skip, chunk_size=args.chunk)
    e2e_local = time.perf_counter() - t0
    e2e_s = max_over_ranks(e2e_local)
    barrier()
    assert c2["checksum"] == cnt["checksum"] and c2["lines"] == cnt["lines"], "the driver's output changed between steps"
    prof_e2e = ctx.profile()
    e2e_value = q_total * args.steps / e2e_s

    # ---- device-ABI leg (rtx_classify_batch, page-locked input and result buffers reused from step to step) -----------------
    reps_a = max(1, min(args.steps, 3))
    res_buf = ctx.pinned_results(nq, max(nq * 8 + 64, n_results + n_results // 4 + 64))
    ctx.classify(off_p, codes_p, eo_p, eids_p, skip_exact=skip, out=res_buf)
    ctx.profile_reset()
    barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps_a):
        out = ctx.classify(off_p, codes_p, eo_p, eids_p, skip_exact=skip, out=res_buf)
    abi_s = max_over_ranks(time.perf_counter() - t0)
    barrier()
    clocks = sampler.stop()  # polled from the start of the device-resident leg to the end of the last timed leg
    prof_abi = ctx.profile()
    assert len(out.first_ref) == n_results

    # ---- roofline of the dominant kernel (hit count) ----------------------------------------------------------
    peak, peak_src = measured_peaks()
    hc = prof["hitcount"]
    n_launch = max(hc["launches"], 1)
    hc_ms = hc["total_ms"] / n_launch
    hc_s = hc_ms * 1e-3
    bitrow_bytes = prof["bitrow_bytes"] / n_launch      # SM side: every selected bit-row slice once per query + the count vectors
    csr_bytes = prof["csr_equiv_bytes"] / n_launch      # what the reference's CSR walk would move (SURVEY 8d primary figure)
    q_per_launch = nq * reps_k / n_launch
    # compulsory HBM traffic of one launch: the bit matrix once (L2 blocking keeps a tile group's slice on chip while all queries of
    # the launch pass over it) + the u16 count vector of every query, written once
    compulsory = ctx.index_bitrow_bytes + q_per_launch * ctx.shard_refs * 2
    sm_mhz = clocks.get("sm_mhz") or 1965.0
    n_sms = torch.cuda.get_device_properties(local_rank).multi_processor_count
    tj_all = {}
    tpath = os.path.join(ROOT, "profiles", "hitcount_traffic.json")
    if os.path.exists(tpath):
        try:
            tj_all = json.load(open(tpath))
        except Exception:
            tj_all = {}
    tj = tj_all.get(name, {})
    dp = tj_all.get("datapath", {})
    # The limiter ncu names is the SM's memory front end, not HBM: the kernel streams scattered 256-byte slices of L2-resident bit rows
    # through the L1 (fill + read-out).  Its ceiling is MEASURED: the same access pattern with no arithmetic at all
    # (tools/micro/smem_tma_probe.cu, profiles/r2_datapath_probe.txt), in bytes per clock and SM.
    path_bpc = float(dp.get("ldg_scattered_256B_slices_B_per_clk_per_SM", 71.2))
    path_peak = path_bpc * n_sms * sm_mhz * 1e6 / 1e9  # GB/s at the clock sampled during the run
    achieved = bitrow_bytes / hc_s / 1e9 if hc_s > 0 else 0.0
    # ncu figures of one launch of THIS workload (profiles/hitcount_traffic.json), DRAM bytes scaled to the live launch by its row-slice bytes
    scale = (bitrow_bytes / tj["bitrow_bytes_per_launch"]) if tj.get("bitrow_bytes_per_launch") else None
    traffic = tj["dram_bytes_per_launch"] * scale if scale and tj.get("dram_bytes_per_launch") else None
    kernel_ms = {k: prof[k]["total_ms"] / reps_k for k in ("kmers", "hitcount", "fixup", "prob", "prefix", "walk")}
    roofline = {
        "kernel": hit_kernel,
        "bound": "sm-l1 (L2 -> L1 fill -> register path of scattered 256-byte bit-row slices; ncu: L1 data pipe %s %%, alu pipe %s %%, DRAM %s of peak) -- "
                 "not hbm: the bit matrix is L2-blocked, see `hbm` and `dram`" % (tj.get("l1_data_pipe_pct", "?"), tj.get("alu_pipe_pct", "?"),
                                                                                   ("%.0f %%" % (100 * traffic / hc_s / 1e9 / peak)) if traffic and hc_s > 0 else "?"),
        "achieved": achieved, "peak": path_peak, "unit": "GB/s", "frac": achieved / path_peak if path_peak > 0 else None,
        "peak_source": "measured ceiling of the path: %.1f B/clk/SM x %d SMs x %.0f MHz (%s)" % (path_bpc, n_sms, sm_mhz, dp.get("source", "default")),
        "algorithmic_bytes_per_launch": bitrow_bytes,
        "algorithmic_bytes_note": "K_q * row_words * 4 + 2 * n_pad per query (DESIGN 4): every selected bit-row slice enters an SM once per query",
        "traffic": traffic,
        "launch_ms": hc_ms, "launches_per_step": n_launch / reps_k, "queries_per_launch": q_per_launch,
        "timed": "kernels serialised, one CUDA event pair per launch on the launching stream (RTX_OPT_PROFILE)",
        "ncu": {k: tj.get(k) for k in ("kernel_symbol", "launch_ms_ncu", "alu_pipe_pct", "l1_data_pipe_pct", "lts_pct", "l1_hit_pct", "l2_hit_pct", "warps_active_pct",
                                       "registers", "source")} if tj else None,
        "hbm": {"bound": "hbm", "algorithmic_bytes_per_launch": compulsory, "achieved": compulsory / hc_s / 1e9 if hc_s > 0 else None, "peak": peak,
                "unit": "GB/s", "frac": compulsory / hc_s / 1e9 / peak if hc_s > 0 else None, "peak_source": peak_src,
                "note": "compulsory traffic: bit matrix once per launch + 2*N bytes of counts per query"},
        "dram": ({"bytes_per_launch": traffic, "gbs": traffic / hc_s / 1e9, "frac_of_peak": traffic / hc_s / 1e9 / peak,
                  "x_compulsory": traffic / compulsory, "source": tj.get("source")} if traffic and hc_s > 0 else None),
        "csr_equivalent": {"bytes_per_launch": csr_bytes, "gbs": csr_bytes / hc_s / 1e9 if hc_s > 0 else None,
                           "note": "4*hits+2*N per query: what the reference's CSR walk would move (SURVEY 8d primary figure)"},
        "serial_ms_per_step": serial_ms, "kernel_ms_per_step": kernel_ms,
        "kernel_share_of_step": {k: v / serial_ms for k, v in kernel_ms.items()} if serial_ms > 0 else None,
    }

    launches = sum(prof_main[k]["launches"] for k in capi.KERNEL_NAMES)
    part = "queries split evenly over the ranks" if scaling == "strong" else f"{q_per_rank} queries per GPU"
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "u32 bit-planes/u16 counts/f64",
            "data": "synthetic",
            "config": {"workload": f"{name}: {ds.n_refs} {kind_name} refs x {ref_len} bp (6-rank lineages) x {q_total} queries, index replicated, {part}"
                                   + (", --skip-exact-matches" if skip else ""),
                       "queries_per_rank": nq,
                       "l2": "no flush needed: bit rows %.0f MB + count vectors %.0f MB per step >> 126 MB L2" % (
                           ctx.index_bytes / 1e6, nq * ctx.shard_refs * 2 / 1e6),
                       "sub_batch": sub_batch, "pipeline": bool(args.pipeline > 0),
                       "tree_build_s": round(t_tree, 2), "index_upload_s": round(t_upload, 2), "results_per_step": int(sum_over_ranks(n_results))},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": prof_e2e["h2d_bytes"] // args.steps,
                    "d2h_bytes_per_step": prof_e2e["d2h_bytes"] // args.steps, "ms_per_step": 1e3 * e2e_s / args.steps,
                    "through": "rxh_raxtax (drop-in for raxtax::raxtax, raxtax.rs:14-97): pageable host query arrays -> exact-match lookup, de-duplication, "
                               "H2D, kernels, D2H, formatting of every result line, per-query hand-off to rxh_count_sender / rxh_count_logger",
                    "result_lines_per_step": cnt["lines"], "result_bytes_per_step": cnt["primary_bytes"], "log_lines_per_step": cnt["log_lines"],
                    "frac_of_device_resident": e2e_value / value},
            "e2e_device_abi": {"value": q_total * reps_a / abi_s, "unit": UNIT, "steps": reps_a, "h2d_bytes_per_step": prof_abi["h2d_bytes"] // reps_a,
                               "d2h_bytes_per_step": prof_abi["d2h_bytes"] // reps_a, "through": "rtx_classify_batch, page-locked host buffers"},
            "gpu_launches": int(launches), "roofline": roofline}

    # ---- reference-sharded check (N > 1): the same references cut into N shards, NCCL collectives inside the device library ------
    if world > 1 and not args.no_sharded:
        from raxtax_b200 import bench_sharded

        n_sh = min(16384, q_per_rank)  # rank 0's slice starts at query 0: its unsharded results above are the expected lines
        rec, _ = bench_sharded.sharded_leg(ctx, tree, ds, n_sh, rank, world, max(1, min(args.steps, 5)), skip, dist, barrier, max_over_ranks,
                                           expect=res if rank == 0 else None)
        if rank == 0:
            assert rec["queries_differing_from_unsharded"] <= max(2, n_sh // 1000), f"reference-sharded run differs from the unsharded one on {rec['queries_differing_from_unsharded']} queries"
        line["sharded"] = rec

    # ---- CPU baseline beside it (rank 0, N = 1 only) -----------------------------------------------------------------
    if world == 1 and not args.no_cpu_baseline:
        ref = CpuReference(ds, skip)
        n_sample, chunk = ref.plan(q_total, cores, 20.0, args.cpu_sample)
        secs = ref.run(n_sample, cores, chunk)
        line["cpu_baseline"] = {"value": n_sample / secs, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"first {n_sample} queries of the same workload (chunks of {chunk}), all {cores} host threads, {secs:.1f} s; C++ port of "
                                          "raxtax.rs / prob.rs / lineage.rs with flat count-indexed histogram tables (O(1) per reference like the reference's ahash "
                                          "maps); the Rust reference cannot be built here (no cargo / rustc)"}
        # the round-1 statement kept its histogram in an ordered std::map (O(log D) per reference): timed once beside it
        n_small = max(cores, n_sample // 4 // cores * cores)
        ref.orc.set_flat_hist(False)
        s_map = ref.run(n_small, cores, max(1, n_small // cores))
        ref.orc.set_flat_hist(True)
        s_flat = ref.run(n_small, cores, max(1, n_small // cores))
        line["cpu_baseline"]["std_map_variant"] = {"value": n_small / s_map, "flat_value_same_sample": n_small / s_flat, "sample": f"first {n_small} queries"}
    if args.dump_outputs:  # res: the device-resident leg's last timed step, this rank's slice of the queries
        if world == 1:
            dump_outputs(res, args.dump_outputs)
        else:
            dump_outputs(res, os.path.join(args.dump_outputs, f"rank{rank}"), DUMP_BYTES // world, first_query=q0)
    if rank == 0:
        emit(line)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
