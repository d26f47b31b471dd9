"""GPU micro-benchmark: hit-count kernel time on a workload for each geometry.

usage: sweep_hitcount.py [workload] [configs]     configs = comma-separated words of letter+number fields, e.g.  G16,G8S2048,G1M4
   G = RTX_OPT_HITCOUNT_GROUP (queries per CTA; 1 = single-query kernel), M = RTX_OPT_HITCOUNT_MAX_TILES,
   S = RTX_OPT_SUB_BATCH (queries per device sub-batch), W = RTX_OPT_WALK_VARIANT, P = RTX_OPT_PIPELINE (two-stream sub-batch pipeline)
   Every configuration's histograms are compared with the first one's (bit-exact).
"""
import json
import os
import re
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

from raxtax_b200 import capi, synth

name = sys.argv[1] if len(sys.argv) > 1 else "c2"
configs = sys.argv[2].split(",") if len(sys.argv) > 2 else ["G1", "G16", "G8", "G4"]
nq = int(sys.argv[3]) if len(sys.argv) > 3 else None
ds = synth.generate(name, n_queries=nq, measure=False)
tree = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes)
ctx = capi.Context(0)
ctx.upload_tree(tree)
eo, eids = tree.exact_batch(ds.query_off, ds.query_codes)
ctx.batch_upload(ds.query_off, ds.query_codes, eo, eids)
OPT = {"G": capi.RTX_OPT_HITCOUNT_GROUP, "M": capi.RTX_OPT_HITCOUNT_MAX_TILES, "S": capi.RTX_OPT_SUB_BATCH, "W": capi.RTX_OPT_WALK_VARIANT,
       "P": capi.RTX_OPT_PIPELINE}
ref = None
ref_counts = None
n_chk = min(192, ds.n_queries)
chk_off = ds.query_off[: n_chk + 1]
chk_codes = ds.query_codes[: int(chk_off[-1])]
chk_eo, chk_eids = tree.exact_batch(chk_off, chk_codes)
for cfg in configs:
    f = {k: int(v) for k, v in re.findall(r"([GMSWP])(\d+)", cfg)}
    for k, o in OPT.items():
        ctx.set_option(o, f.get(k, 0))
    ctx.batch_upload(ds.query_off, ds.query_codes, eo, eids)  # the sub-batch size is fixed at upload time
    ctx.set_option(capi.RTX_OPT_PROFILE, 0)
    ctx.batch_run()
    ctx.synchronize()
    t0 = time.perf_counter()
    for _ in range(3):
        ctx.batch_run()
    ctx.synchronize()
    pass_ms = (time.perf_counter() - t0) / 3 * 1e3  # whole pass, kernels overlapping as they do in production
    ctx.set_option(capi.RTX_OPT_PROFILE, 1)
    ctx.profile_reset()
    for _ in range(3):
        ctx.batch_run()
    out = ctx.batch_download(taps=("hist",))
    p = ctx.profile()
    if ref is None:
        ref = out.hist.copy()
    ms = p["hitcount"]["total_ms"] / 3  # per pass over the whole batch (a pass is several launches when sub-batched)
    gbs = p["bitrow_bytes"] / 3 / ms / 1e6
    small = ctx.classify(chk_off, chk_codes, chk_eo, chk_eids, taps=("counts",))  # the count vectors themselves (the layout inside a tile is the kernel's business)
    if ref_counts is None:
        ref_counts = small.counts.copy()
    counts_same = bool(np.array_equal(small.counts, ref_counts))
    print(json.dumps(dict(cfg=cfg, pass_ms=round(pass_ms, 3), kernel=ctx.hitcount_kernel_name(), counts_identical=counts_same, hitcount_ms=round(ms, 3), bitrow_GBps=round(gbs, 1), prob_ms=round(p["prob"]["total_ms"] / 3, 3),
                          prefix_ms=round(p["prefix"]["total_ms"] / 3, 3), walk_ms=round(p["walk"]["total_ms"] / 3, 3),
                          hist_identical=bool(np.array_equal(out.hist, ref)))), flush=True)
