"""Reference-sharded leg of bench.py (BASELINE config 5 and the sharded check of the multi-GPU default run): the references are cut
into `world` contiguous shards of the lineage-sorted order, every rank holds one shard and sees every query, the per-query count
histograms are all-reduced and the straddler records all-gathered by NCCL inside the device library (rtx_shard_run), the result lines
are gathered and merged on rank 0 (rtx_shard_gather)."""
from __future__ import annotations

import time

import numpy as np

from . import capi


def broadcast_unique_id(dist, rank):
    import torch

    uid = capi.Context.comm_unique_id() if rank == 0 else bytes(128)
    t = torch.tensor(list(uid), dtype=torch.uint8, device="cuda")
    dist.broadcast(t, src=0)
    return bytes(t.cpu().tolist())


def sharded_leg(ctx, tree, ds, n_queries, rank, world, steps, skip, dist, barrier, max_over_ranks, expect=None, sub_batch=0):
    """Classifies the first n_queries queries of ds on `world` reference shards; returns the record for the bench line (rank 0) and the
    ClassifyOutput of the last timed step (the merged lines on rank 0), and leaves ctx holding the sharded index.  expect = ClassifyOutput
    of the same queries from an unsharded context: compared line by line."""
    import torch

    N = tree.num_tips
    cuts = np.array([N * r // world for r in range(world)] + [N], np.uint64)
    ctx.comm_init(broadcast_unique_id(dist, rank), rank, world)
    t0 = time.time()
    ctx.upload_tree_sharded(tree, world, rank, cuts)
    t_upload = time.time() - t0
    off = np.ascontiguousarray(ds.query_off[: n_queries + 1], np.uint64)
    codes = ds.query_codes[: int(off[-1])]
    eo, eids = tree.exact_batch(off, codes)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
    off_p, codes_p, eo_p, eids_p = pin(off), pin(codes), pin(eo), pin(eids if len(eids) else np.zeros(1, np.uint32))
    if sub_batch:
        ctx.set_option(capi.RTX_OPT_SUB_BATCH, sub_batch)
    out = None
    for _ in range(2):
        out = ctx.classify(off_p, codes_p, eo_p, eids_p, skip_exact=skip, shard_root=0)
    n_diff = None
    if expect is not None and rank == 0:
        # per query: the same lines (first reference, levels, confidences bit for bit, signals to 1e-9) as the unsharded context gave.
        # Queries whose probability profile is exactly flat (K = 0: every node confidence is size/N, sitting ON rounding boundaries and
        # exact ties) may legitimately differ -- the sharded sums add the same numbers in another order (tools/shard_diff.py judges such
        # queries against the CPU restatement: both outcomes acceptable); they are counted, not hidden.
        eb, gb = expect.result_begin[: n_queries + 1].astype(np.int64), out.result_begin.astype(np.int64)
        bad = (gb[1:] - gb[:-1]) != (eb[1:] - eb[:-1])
        ok_q = np.nonzero(~bad)[0]
        if len(ok_q):
            cnt = (eb[1:] - eb[:-1])[ok_q]
            qi = np.repeat(ok_q, cnt)                                   # query of every compared line
            k = np.arange(len(qi)) - np.repeat(np.cumsum(cnt) - cnt, cnt)  # position of the line within its query
            ei, gi = eb[qi] + k, gb[qi] + k
            lev = np.arange(expect.confidence.shape[1])[None, :] < expect.n_levels[ei][:, None]
            line_ok = ((out.first_ref[gi] == expect.first_ref[ei]) & (out.n_levels[gi] == expect.n_levels[ei])
                       & np.all((out.confidence[gi] == expect.confidence[ei]) | ~lev, axis=1) & (np.abs(out.local_signal[gi] - expect.local_signal[ei]) <= 1e-9))
            bad[np.unique(qi[~line_ok])] = True
        bad |= np.abs(out.global_signal - expect.global_signal[:n_queries]) > 1e-9
        n_diff = int(bad.sum())
    ctx.set_option(capi.RTX_OPT_PROFILE, 1)
    ctx.classify(off_p, codes_p, eo_p, eids_p, skip_exact=skip, shard_root=0)
    ctx.profile_reset()
    reps_p = max(1, min(steps, 2))
    for _ in range(reps_p):
        ctx.classify(off_p, codes_p, eo_p, eids_p, skip_exact=skip, shard_root=0)
    prof = ctx.profile()
    ctx.set_option(capi.RTX_OPT_PROFILE, 0)
    ctx.profile_reset()
    barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        out = ctx.classify(off_p, codes_p, eo_p, eids_p, skip_exact=skip, shard_root=0)
    secs = max_over_ranks(time.perf_counter() - t0)
    barrier()
    prof_t = ctx.profile()
    launches = sum(prof_t[k]["launches"] for k in capi.KERNEL_NAMES)
    rec = {"value": n_queries * steps / secs, "unit": "queries/s", "n_ranks": world, "queries": n_queries, "steps": steps, "ms_per_step": 1e3 * secs / steps,
           "references": int(N), "references_per_shard": int(N // world), "sub_batch": ctx.sub_batch, "index_upload_s": round(t_upload, 2),
           "result_lines": int(out.result_begin[-1]) if rank == 0 else None,
           "through": "rtx_shard_classify on every rank (page-locked host buffers): H2D, k-mers, per sub-batch hit counts | ncclAllReduce(u32 sum) of the "
                      "histogram rows | P(count), prefixes, straddler records | ncclAllGather | combine + walk (collectives and tail kernels of sub-batch i "
                      "under the hit counting of sub-batch i+1), then ncclSend/Recv of the result lines to rank 0, device merge, D2H",
           "phase_ms_per_step_rank0": {k: prof[k]["total_ms"] / reps_p for k in ("kmers", "hitcount", "fixup", "allreduce", "prob", "prefix", "shard", "allgather", "walk", "gather")},
           "phase_note": "CUDA-event durations per launch on the launching stream; allreduce / allgather / gather are the NCCL calls (they include waiting for the "
                         "slowest rank), and they overlap the next sub-batch's hit counting on the other stream, so the phases add up to more than a step",
           "collective_bytes_per_step_rank0": {"allreduce": prof["allreduce_bytes"] // reps_p, "allgather": prof["allgather_bytes"] // reps_p,
                                               "gather": prof["gather_bytes"] // reps_p},
           "h2d_bytes_per_step": prof_t["h2d_bytes"] // steps, "d2h_bytes_per_step": prof_t["d2h_bytes"] // steps, "gpu_launches": int(launches),
           "queries_differing_from_unsharded": n_diff,
           "identical_note": "compared line by line with rank 0's unsharded results of the same queries; flat-profile (K = 0) queries sit on exact "
                             "ties / rounding boundaries and may differ (DESIGN 2, tools/shard_diff.py)"}
    return rec, out


def run(args, rank, local_rank, world, barrier, max_over_ranks, load_workload, ClockSampler, measured_peaks, METRIC, UNIT):
    """bench.py --workload c5: 8 M references (1 M per shard at 8 ranks), a bounded job of --queries queries (default 131 072).
    Returns the bench line and the ClassifyOutput of the last timed step (every query's lines on rank 0)."""
    import torch
    import torch.distributed as dist

    from . import synth

    name = "c5"
    nq = args.queries
    ds = load_workload(name, nq, rank, barrier)
    t0 = time.time()
    tree = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes)
    t_tree = time.time() - t0
    ctx = capi.Context(local_rank)
    sampler = ClockSampler(local_rank)
    sampler.start()
    if world == 1:
        # one rank: nothing to shard or exchange -- the whole index on this GPU (66 GB of bit rows), the ordinary path
        ctx.upload_tree(tree)
        off = np.ascontiguousarray(ds.query_off[: nq + 1], np.uint64)
        codes = ds.query_codes[: int(off[-1])]
        eo, eids = tree.exact_batch(off, codes)
        for _ in range(2):
            ctx.classify(off, codes, eo, eids)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            out = ctx.classify(off, codes, eo, eids)
        secs = time.perf_counter() - t0
        rec = {"value": nq * args.steps / secs, "ms_per_step": 1e3 * secs / args.steps, "n_ranks": 1, "queries": nq, "through": "rtx_classify_batch, unsharded (one rank)",
               "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "gpu_launches": 0}
    else:
        rec, out = sharded_leg(ctx, tree, ds, nq, rank, world, args.steps, False, dist, barrier, max_over_ranks, sub_batch=args.sub_batch)
    clocks = sampler.stop()
    line = {"metric": METRIC, "value": rec["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": 2, "ms_per_step": rec["ms_per_step"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32 bit-planes/u16 counts/f64", "data": "synthetic",
            "config": {"workload": f"c5: {ds.n_refs} COI-like refs x {synth.CONFIGS[name][2]} bp, reference-sharded over {world} ranks, bounded job of {nq} queries "
                                   "(every rank sees every query)", "tree_build_s": round(t_tree, 2)},
            "clocks": clocks,
            "e2e": {"value": rec["value"], "unit": UNIT, "h2d_bytes_per_step": rec["h2d_bytes_per_step"], "d2h_bytes_per_step": rec["d2h_bytes_per_step"],
                    "through": rec["through"]},
            "gpu_launches": rec["gpu_launches"], "sharded": rec}
    ctx.close()
    return line, out
