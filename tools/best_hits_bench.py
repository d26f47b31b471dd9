"""What reporting each query's best hits (RTX_OPT_BEST_HITS) costs, on the synthetic workloads, on one GPU, in one process.

For each workload (default c2 and c3) three device-resident legs run on the same index and batch, alternating, `--rounds` times:
  T0    best hits off (the classification alone)
  T10   best_hits = 10
  T64   best_hits = 64
and the script checks:
  * the last download of every T > 0 leg: result lines, n_kmers and global signals bit-identical to T0;
  * on a sample of `--sample` queries classified with every tap: result lines, signals and all four taps of T = 10 and 64
    bit-identical to T = 0, and the hits equal to the numpy selection over tap_counts (count descending, id ascending, first T of
    the references with count >= 1) -- and equal to the hits the full-batch legs returned for the same queries.
It reports the median ms per step of every leg (batch resident in HBM, CUDA events on the context's stream), the overhead over T0,
and the card's name and power limit before and after.

  python tools/best_hits_bench.py [--workloads c2,c3] [--steps 3] [--warmup 1] [--rounds 3] [--sample 300] [--out FILE.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

LEGS = {"T0": 0, "T10": 10, "T64": 64}
TAPS = ("counts", "hist", "kmers", "probs")


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return out.stdout.strip().split("\n")[0] if out.returncode == 0 else "unknown"


def same_lines(a, b):
    return bool(np.array_equal(a.result_begin, b.result_begin) and np.array_equal(a.first_ref, b.first_ref)
                and np.array_equal(a.n_levels, b.n_levels) and np.array_equal(a.confidence, b.confidence)
                and np.array_equal(a.local_signal, b.local_signal) and np.array_equal(a.global_signal, b.global_signal)
                and np.array_equal(a.n_kmers, b.n_kmers))


def numpy_hits(counts, T):
    """Per row: the ids with count >= 1 by (count desc, id asc), the first T."""
    out = []
    for row in counts:
        nz = np.nonzero(row)[0]
        sel = nz[np.lexsort((nz, -row[nz].astype(np.int64)))][:T]
        out.append((sel, row[sel]))
    return out


def hits_mismatches(hits, want, rows=None):
    """Queries whose device hits (n, ref, count) differ from want[i] = (ids, counts); rows: which device rows want[i] belongs to."""
    n, ref, cnt = hits
    bad = 0
    for i, (ids, c) in enumerate(want):
        q = i if rows is None else rows[i]
        k = int(n[q])
        bad += int(k != len(ids) or not np.array_equal(ref[q, :k], ids) or not np.array_equal(cnt[q, :k], c))
    return bad


def run_workload(name, args, capi, synth, load_workload, torch):
    ds = load_workload(name, synth.CONFIGS[name][1])
    tree = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes)
    ctx = capi.Context(0)
    ctx.upload_tree(tree)
    off = np.ascontiguousarray(ds.query_off - ds.query_off[0], np.uint64)
    codes = np.ascontiguousarray(ds.query_codes, np.uint8)
    eo, eids = tree.exact_batch(off, codes)
    nq = len(off) - 1
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", 0))
    times = {k: [] for k in LEGS}
    outs = {}
    for r in range(args.rounds):
        for leg, T in LEGS.items():
            ctx.batch_upload(off, codes, eo, eids, best_hits=T)
            for _ in range(args.warmup):
                ctx.batch_run()
            ctx.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(stream)
            for _ in range(args.steps):
                ctx.batch_run()
            ev1.record(stream)
            ctx.synchronize()
            times[leg].append(ev0.elapsed_time(ev1) / args.steps)
            if r == args.rounds - 1:
                outs[leg] = ctx.batch_download()
    ms = {k: float(np.median(v)) for k, v in times.items()}
    # the sample: every tap, T = 0 against T > 0, hits against numpy and against the full-batch legs
    rng = np.random.default_rng(12345)
    pick = np.sort(rng.choice(nq, min(args.sample, nq), replace=False))
    s_seqs = [codes[int(off[q]): int(off[q + 1])] for q in pick]
    s_off = np.zeros(len(pick) + 1, np.uint64)
    s_off[1:] = np.cumsum([len(s) for s in s_seqs])
    s_codes = np.concatenate(s_seqs)
    s_eo, s_eids = tree.exact_batch(s_off, s_codes)
    s0 = ctx.classify(s_off, s_codes, s_eo, s_eids, taps=TAPS)
    checks = {}
    for leg, T in LEGS.items():
        if not T:
            continue
        st = ctx.classify(s_off, s_codes, s_eo, s_eids, taps=TAPS, best_hits=T)
        want = numpy_hits(s0.counts, T)
        checks[leg] = {
            "batch_lines_signals_identical_to_T0": same_lines(outs[leg], outs["T0"]),
            "sample_lines_signals_identical_to_T0": same_lines(st, s0),
            "sample_taps_identical_to_T0": all(bool(np.array_equal(getattr(st, t), getattr(s0, t))) for t in TAPS),
            "sample_queries": int(len(pick)),
            "sample_hits_differing_from_numpy": hits_mismatches(st.best_hits, want),
            "batch_hits_differing_from_numpy": hits_mismatches(outs[leg].best_hits, want, pick),
            "sample_queries_with_T_hits": int((st.best_hits[0] == T).sum()),
        }
    ctx.close()
    return {
        "workload": name, "n_refs": ds.n_refs, "n_queries": nq, "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds,
        "ms_per_step": ms, "ms_per_step_all_rounds": times,
        "overhead_over_T0": {k: ms[k] / ms["T0"] - 1.0 for k in LEGS if k != "T0"},
        "checks": checks,
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--workloads", default="c2,c3")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--sample", type=int, default=300)
    ap.add_argument("--out", default="", help="also write the JSON report here")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("best_hits_bench.py measures on a CUDA device; none is available")
    from bench import load_workload
    from raxtax_b200 import capi, synth

    report = {"gpu": gpu_info(), "time": time.strftime("%Y-%m-%d %H:%M:%S"), "workloads": []}
    for name in args.workloads.split(","):
        r = run_workload(name.strip(), args, capi, synth, load_workload, torch)
        report["workloads"].append(r)
        print(json.dumps(r), flush=True)
    report["gpu_after"] = gpu_info()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)
    print(json.dumps({"gpu": report["gpu"], "gpu_after": report["gpu_after"]}))
    ok = all(c["batch_lines_signals_identical_to_T0"] and c["sample_lines_signals_identical_to_T0"] and c["sample_taps_identical_to_T0"]
             and c["sample_hits_differing_from_numpy"] == 0 and c["batch_hits_differing_from_numpy"] == 0
             for w in report["workloads"] for c in w["checks"].values())
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
