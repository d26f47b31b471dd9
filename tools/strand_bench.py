"""--strand both against plus mode on the synthetic workloads, on one GPU, in one process.

For each workload (default c2 and c3) four device-resident legs run on the same index, alternating, `--rounds` times:
  plus            the queries as generated
  plus_reversed   every query reverse-complemented
  both            the queries as generated, RTX_BOTH_STRANDS
  both_reversed   every query reverse-complemented, RTX_BOTH_STRANDS
and the script checks, query by query (identical lines, first_ref, n_levels and confidences; signals within 1e-12):
  * both_reversed: a query reported `-` gives exactly plus's result of the original query, one reported `+` exactly plus_reversed's
    result, and which one follows the rule M(rc(s)) > M(s) with M taken from the histograms of the two plus legs;
  * both: a query reported `+` gives exactly plus's result (and `-` exactly plus_reversed's), by the same rule.
With --segmax-compare a fifth leg, both_no_segmax, runs the `both` batch on a second context created with RTX_STRAND_SEGMAX=0 (no
per-segment maxima, K4 reads every count) and must give the same results as `both`.
It reports queries/s of every leg (batch resident in HBM, CUDA events on the context's stream, median over the rounds), the
both / plus time ratio, the fraction of each query kind (label suffix |kind0..3) reported `-`, the card's name and power limit.

  python tools/strand_bench.py [--workloads c2,c3] [--steps 3] [--warmup 1] [--rounds 2] [--segmax-compare] [--out FILE.json]
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

SIGNAL_TOL = 1e-12


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return out.stdout.strip().split("\n")[0] if out.returncode == 0 else "unknown"


def top_bucket(hist):
    """M per query: the largest count with a non-empty histogram bucket."""
    nz = hist != 0
    return np.where(nz.any(axis=1), hist.shape[1] - 1 - np.argmax(nz[:, ::-1], axis=1), 0)


def pick_lines(pick, src0, src1):
    """The result lines of src1 where pick, else of src0, in query order: (first_ref, n_levels, confidence, local_signal, line query)."""
    c0, c1 = np.diff(src0.result_begin.astype(np.int64)), np.diff(src1.result_begin.astype(np.int64))
    cnt = np.where(pick, c1, c0)
    begin = np.where(pick, src1.result_begin[:-1].astype(np.int64) + len(src0.first_ref), src0.result_begin[:-1].astype(np.int64))
    within = np.arange(int(cnt.sum())) - np.repeat(np.cumsum(cnt) - cnt, cnt)
    idx = np.repeat(begin, cnt) + within
    cat = lambda a, b: np.concatenate([a, b])
    return (cat(src0.first_ref, src1.first_ref)[idx], cat(src0.n_levels, src1.n_levels)[idx], cat(src0.confidence, src1.confidence)[idx],
            cat(src0.local_signal, src1.local_signal)[idx], cnt)


def check_against(both, pick, src0, src1):
    """Number of queries whose lines in `both` differ from the picked plus-mode lines."""
    first, nlev, conf, local, cnt = pick_lines(pick, src0, src1)
    got_cnt = np.diff(both.result_begin.astype(np.int64))
    if not np.array_equal(cnt, got_cnt):
        return int((cnt != got_cnt).sum()), "line counts differ"
    q_of_line = np.repeat(np.arange(len(cnt)), cnt)
    bad_line = ((both.first_ref != first) | (both.n_levels != nlev) | np.any(both.confidence != conf, axis=1)
                | (np.abs(both.local_signal - local) > SIGNAL_TOL))
    bad = np.zeros(len(cnt), bool)
    bad[q_of_line[bad_line]] = True
    bad |= np.abs(both.global_signal - np.where(pick, src1.global_signal, src0.global_signal)) > SIGNAL_TOL
    bad |= both.n_kmers != np.where(pick, src1.n_kmers, src0.n_kmers)
    return int(bad.sum()), ""


def run_workload(name, args, capi, synth, load_workload, torch):
    ds = load_workload(name, synth.CONFIGS[name][1])
    tree = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes)
    ctx = capi.Context(0)
    ctx.upload_tree(tree)
    off = np.ascontiguousarray(ds.query_off - ds.query_off[0], np.uint64)
    codes = np.ascontiguousarray(ds.query_codes, np.uint8)
    rev = synth.reverse_complement_batch(off, codes)
    legs = {
        "plus": (codes, tree.exact_batch(off, codes), False),
        "plus_reversed": (rev, tree.exact_batch(off, rev), False),
        "both": (codes, tree.exact_batch_both_strands(off, codes), True),
        "both_reversed": (rev, tree.exact_batch_both_strands(off, rev), True),
    }
    ctxs = {leg: ctx for leg in legs}
    if args.segmax_compare:
        os.environ["RTX_STRAND_SEGMAX"] = "0"
        ctx_ns = capi.Context(0)
        del os.environ["RTX_STRAND_SEGMAX"]
        ctx_ns.upload_tree(tree)
        legs["both_no_segmax"] = legs["both"]
        ctxs["both_no_segmax"] = ctx_ns
    times = {k: [] for k in legs}
    outs = {}
    for r in range(args.rounds):
        for leg, (c, (eo, eids), both) in legs.items():
            cx = ctxs[leg]
            stream = torch.cuda.ExternalStream(cx.stream, device=torch.device("cuda", 0))
            cx.batch_upload(off, c, eo, eids, both_strands=both)
            for _ in range(args.warmup):
                cx.batch_run()
            cx.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(stream)
            for _ in range(args.steps):
                cx.batch_run()
            ev1.record(stream)
            cx.synchronize()
            times[leg].append(ev0.elapsed_time(ev1) / args.steps)
            if r == args.rounds - 1:
                o = cx.batch_download(taps=("hist",) if not both else ())
                if o.hist is not None:
                    o.M = top_bucket(o.hist)
                    o.hist = None
                outs[leg] = o
    nq = len(off) - 1
    ms = {k: float(np.median(v)) for k, v in times.items()}
    plus, plus_rev, both, both_rev = outs["plus"], outs["plus_reversed"], outs["both"], outs["both_reversed"]
    # as generated: `-` iff M(rc(s)) = M of the reversed leg > M(s); reversed input: `-` iff M of the original > M of the reversed
    rule_gen = (plus_rev.M > plus.M).astype(np.uint8)
    rule_rev = (plus.M > plus_rev.M).astype(np.uint8)
    bad_gen, why_gen = check_against(both, both.strand.astype(bool), plus, plus_rev)
    bad_rev, why_rev = check_against(both_rev, both_rev.strand.astype(bool), plus_rev, plus)
    kinds = np.array([int(l.rsplit("|kind", 1)[1]) if "|kind" in l else -1 for l in ds.query_labels])
    minus = {}
    for leg, o in (("both", both), ("both_reversed", both_rev)):
        minus[leg] = {f"kind{k}": float(o.strand[kinds == k].mean()) for k in sorted(set(kinds.tolist())) if (kinds == k).any()}
        minus[leg]["all"] = float(o.strand.mean())
    checks_extra = {}
    if args.segmax_compare:
        ns = outs["both_no_segmax"]
        checks_extra["both_no_segmax_identical_to_both"] = bool(
            np.array_equal(ns.strand, both.strand) and np.array_equal(ns.result_begin, both.result_begin) and np.array_equal(ns.first_ref, both.first_ref)
            and np.array_equal(ns.confidence, both.confidence) and np.array_equal(ns.local_signal, both.local_signal)
            and np.array_equal(ns.global_signal, both.global_signal))
        ctxs["both_no_segmax"].close()
    ctx.close()
    return {
        "workload": name, "n_refs": ds.n_refs, "n_queries": nq, "steps": args.steps, "rounds": args.rounds,
        "ms_per_step": ms, "qps": {k: nq / (v / 1e3) for k, v in ms.items()},
        "ratio_both_over_plus": ms["both"] / ms["plus"], "ratio_both_reversed_over_plus": ms["both_reversed"] / ms["plus"],
        "fraction_minus": minus,
        "checks": {
            "both_strand_follows_rule": bool(np.array_equal(both.strand, rule_gen)),
            "both_reversed_strand_follows_rule": bool(np.array_equal(both_rev.strand, rule_rev)),
            "both_queries_differing_from_plus_legs": bad_gen, "both_reversed_queries_differing_from_plus_legs": bad_rev,
            "notes": " ".join(x for x in (why_gen, why_rev) if x), **checks_extra,
        },
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--workloads", default="c2,c3")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--segmax-compare", action="store_true", help="add the both_no_segmax leg (RTX_STRAND_SEGMAX=0)")
    ap.add_argument("--out", default="", help="also write the JSON report here")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("strand_bench.py measures on a CUDA device; none is available")
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
    ok = all(w["checks"]["both_strand_follows_rule"] and w["checks"]["both_reversed_strand_follows_rule"]
             and w["checks"]["both_queries_differing_from_plus_legs"] == 0 and w["checks"]["both_reversed_queries_differing_from_plus_legs"] == 0
             and w["checks"].get("both_no_segmax_identical_to_both", True) for w in report["workloads"])
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
