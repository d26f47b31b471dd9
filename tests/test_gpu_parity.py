"""GPU parity tests (run on the B200 box with `-m gpu`): the CUDA path, called through the C ABI, against the
CPU oracle on the same seeded inputs, against the committed golden fixtures and through size-independent properties."""
import os

import numpy as np
import pytest

from raxtax_b200 import capi, synth
from tests import parity
from tests.test_oracle_kats import KMER_KAT_CODES, KMER_KAT_EXPECTED, REF_FASTA_KMERS, REF_FASTA_STR_PARSER

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


def _pack(orc, seqs):
    return orc.pack_sequences([np.asarray(s, np.uint8) for s in seqs])


def _run_both(orc, ctx, ds_or_tuple, skip=False, raw=False, sub_batch=0, variant=capi.RTX_HITCOUNT_BITROWS, threads=4):
    """-> (oracle dict, device ClassifyOutput, oracle tree, host tree)"""
    if isinstance(ds_or_tuple, tuple):
        lineages, ref_off, ref_codes, q_off, q_codes = ds_or_tuple
    else:
        ds = ds_or_tuple
        lineages, ref_off, ref_codes, q_off, q_codes = ds.ref_lineages, ds.ref_off, ds.ref_codes, ds.query_off, ds.query_codes
    seqs = [ref_codes[int(ref_off[i]): int(ref_off[i + 1])] for i in range(len(lineages))]
    ot = orc.Tree.new(lineages, seqs)
    ht = capi.Tree.new(lineages, ref_off, ref_codes, eager_kmer_map=variant == capi.RTX_HITCOUNT_CSR)  # the CSR variant walks Tree.k_mer_map itself
    ctx.set_option(capi.RTX_OPT_KEEP_CSR, 1 if variant == capi.RTX_HITCOUNT_CSR else 0)
    ctx.set_option(capi.RTX_OPT_HITCOUNT_VARIANT, variant)
    ctx.set_option(capi.RTX_OPT_SUB_BATCH, sub_batch)
    ctx.upload_tree(ht)
    eo, eids = ht.exact_batch(q_off, q_codes)
    dev = ctx.classify(q_off, q_codes, eo, eids, skip_exact=skip, raw_conf=raw, taps=("counts", "hist", "kmers", "probs"))
    o = ot.classify(q_off, q_codes, skip_exact=skip, raw_conf=raw, threads=threads, chunk_size=16, want_counts=True, want_probs=True,
                    want_kmers=True)
    ctx.set_option(capi.RTX_OPT_HITCOUNT_VARIANT, capi.RTX_HITCOUNT_BITROWS)
    ctx.set_option(capi.RTX_OPT_KEEP_CSR, 0)
    ctx.set_option(capi.RTX_OPT_SUB_BATCH, 0)
    return o, dev, ot, ht


def _assert_integer_parity(o, dev, nq):
    assert np.array_equal(o["K"], dev.n_kmers)
    for q in range(nq):
        K = int(o["K"][q])
        assert np.array_equal(o["kmers"][q, :K], dev.kmers[q, :K]), f"k-mer list of query {q}"
    assert np.array_equal(o["counts"], dev.counts), "hit counts"
    for q in range(nq):
        K = int(o["K"][q])
        assert np.array_equal(parity.hist_from_counts(o["counts"][q], K), dev.hist[q, : K + 1]), f"histogram of query {q}"


PROB_ATOL = 1e-9  # normalised highest-hit probabilities (prob.rs:8-103); north_star tolerance is 1e-6, observed ~1e-13


def _assert_prob_parity(o, dev, nq):
    worst = 0.0
    for q in range(nq):
        dp = dev.probs[q][dev.counts[q].astype(np.int64)]  # gather per reference, as prob.rs:92-95
        worst = max(worst, float(np.max(np.abs(dp - o["probs"][q]))))
    assert worst <= PROB_ATOL, f"probabilities differ from the oracle by {worst:.3e}"
    return worst


def _assert_result_parity(o, dev, ot, nq, max_tolerated_frac=0.05):
    if dev.probs is not None and dev.counts is not None and "probs" in o:
        _assert_prob_parity(o, dev, nq)
    checker = parity.TolerantChecker(ot.flatten(), ot.num_tips)
    ok, tol, bad = parity.compare_batch(o, dev, nq, checker, o["probs"])
    assert not bad, f"{len(bad)} queries differ beyond tie/boundary tolerance, first: {bad[:5]}: oracle={o['results'].for_query(bad[0])} device={dev.for_query(bad[0])}"
    assert tol <= max(1, int(max_tolerated_frac * nq)), f"{tol} of {nq} queries needed tie/boundary tolerance"
    return ok, tol


# ---- reference KATs through the CUDA path ---------------------------------------------------------------------------
def test_kmer_kat_on_device(oracle, ctx):  # utils.rs:245-263
    ht = capi.Tree.from_fasta(REF_FASTA_STR_PARSER)
    ctx.upload_tree(ht)
    off, codes = _pack(oracle, [KMER_KAT_CODES, [1] * 7, [], [8] * 30, [1] * 7 + [15] + [1] * 7])
    dev = ctx.classify(off, codes, taps=("kmers",))
    assert list(dev.n_kmers) == [8, 0, 0, 1, 0]
    assert list(dev.kmers[0, :8]) == KMER_KAT_EXPECTED
    assert dev.kmers[3, 0] == 0xFFFF


@pytest.mark.parametrize("fasta", [REF_FASTA_STR_PARSER, REF_FASTA_KMERS])
def test_parser_kat_databases_classified_like_oracle(oracle, ctx, fasta):  # parser.rs:166-299 databases, self-queries
    ot = oracle.Tree.from_fasta(fasta)
    seqs = [ot.sequence(i) for i in range(ot.num_tips)] + [oracle.map_dna("ATACGCTTTGGGTA"), oracle.map_dna("NNNNNNNNNN")]
    q_off, q_codes = _pack(oracle, seqs)
    r_off, r_codes = _pack(oracle, [ot.sequence(i) for i in range(ot.num_tips)])
    for skip, raw in [(False, False), (True, False), (False, True)]:
        o, dev, ot2, _ = _run_both(oracle, ctx, (ot.lineages, r_off, r_codes, q_off, q_codes), skip=skip, raw=raw)
        _assert_integer_parity(o, dev, len(seqs))
        _assert_result_parity(o, dev, ot2, len(seqs), max_tolerated_frac=1.0)


# ---- seeded synthetic data ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("skip,raw", [(False, False), (True, False), (False, True)])
def test_tiny_dataset_parity(oracle, ctx, skip, raw):
    ds = synth.generate("tiny", measure=False)
    o, dev, ot, _ = _run_both(oracle, ctx, ds, skip=skip, raw=raw)
    _assert_integer_parity(o, dev, ds.n_queries)
    _assert_result_parity(o, dev, ot, ds.n_queries)


def test_small_dataset_parity_and_text_output(oracle, ctx):
    ds = synth.generate("small", measure=False)
    o, dev, ot, ht = _run_both(oracle, ctx, ds)
    _assert_integer_parity(o, dev, ds.n_queries)
    ok, tol = _assert_result_parity(o, dev, ot, ds.n_queries)
    # formatted raxtax.out / raxtax.tsv lines through the host driver vs the oracle's formatting of its own results
    qs = capi.Queries.new(ds.query_labels, ds.query_off, ds.query_codes)
    sent, logs, _ = capi.raxtax(ctx, qs, ht, chunk_size=100, tsv=True)
    assert [s[0] for s in sent] == ds.query_labels
    exp_primary = oracle.format_results(ot, o["results"], ds.query_labels).split("\n")
    exp_tsv = oracle.format_results(ot, o["results"], ds.query_labels, ds.query_off, ds.query_codes, tsv=True).split("\n")
    got_primary = [l for s in sent for l in s[1].split("\n")]
    got_tsv = [l for s in sent for l in s[2].split("\n")]
    if tol == 0:
        assert got_primary == exp_primary
        assert got_tsv == exp_tsv
    else:
        same = sum(a == b for a, b in zip(got_primary, exp_primary))
        assert same >= 0.95 * len(exp_primary)
    # log lines: one Info line per exact match (raxtax.rs:46-48)
    n_exact = int(o["nexact"].sum())
    assert sum(1 for lvl, _ in logs if lvl == 3) == n_exact


def test_small_dataset_skip_exact_sub_batched(oracle, ctx):
    ds = synth.generate("small", measure=False)
    o, dev, ot, _ = _run_both(oracle, ctx, ds, skip=True, sub_batch=37)
    _assert_integer_parity(o, dev, ds.n_queries)
    _assert_result_parity(o, dev, ot, ds.n_queries)


def test_csr_variant_matches_bitrows(oracle, ctx):
    ds = synth.generate("tiny", measure=False)
    o, dev, ot, _ = _run_both(oracle, ctx, ds, variant=capi.RTX_HITCOUNT_CSR)
    _assert_integer_parity(o, dev, ds.n_queries)
    _assert_result_parity(o, dev, ot, ds.n_queries)


def _same_outputs(a, b):
    return (np.array_equal(a.result_begin, b.result_begin) and np.array_equal(a.first_ref, b.first_ref) and np.array_equal(a.n_levels, b.n_levels)
            and np.array_equal(a.confidence, b.confidence) and np.array_equal(a.local_signal, b.local_signal)
            and np.array_equal(a.global_signal, b.global_signal))


@pytest.mark.parametrize("skip", [False, True])
def test_walk_variants_agree(ctx, skip):
    """Level-synchronous walk (default), depth-first walker, and the retry path (log cap forced down so that most queries are
    handed back to the depth-first walker) must produce bit-identical result lists."""
    ds = synth.generate("small", n_queries=512, measure=False)
    ht = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes)
    ctx.upload_tree(ht)
    eo, eids = ht.exact_batch(ds.query_off, ds.query_codes)
    outs = []
    try:
        for variant, cap in ((0, 0), (1, 0), (0, 8), (0, 40)):
            ctx.set_option(capi.RTX_OPT_WALK_VARIANT, variant)
            ctx.set_option(capi.RTX_OPT_WALK_LOG_CAP, cap)
            outs.append(ctx.classify(ds.query_off, ds.query_codes, eo, eids, skip_exact=skip))
    finally:
        ctx.set_option(capi.RTX_OPT_WALK_VARIANT, 0)
        ctx.set_option(capi.RTX_OPT_WALK_LOG_CAP, 0)
    assert len(outs[0].first_ref) >= ds.n_queries
    for o in outs[1:]:
        assert _same_outputs(outs[0], o)


def test_index_built_from_sequences_matches_csr_index(ctx):
    """The device builds its bit rows either from the host's k_mer_map (CSR, tree.rs:41) or -- default, no k_mer_map on the host --
    from the sorted reference sequences themselves (tree.rs:114-123 windowing on the device): same counts, same results."""
    ds = synth.generate("small", n_queries=300, measure=False)
    ht = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes)
    assert not ht.has_kmer_map
    eo, eids = ht.exact_batch(ds.query_off, ds.query_codes)
    ctx.upload_tree(ht)  # sequence path
    a = ctx.classify(ds.query_off, ds.query_codes, eo, eids, taps=("counts", "hist", "kmers"))
    bytes_seq = ctx.index_bytes
    ht.build_kmer_map()
    assert ht.has_kmer_map
    ctx.upload_tree(ht)  # CSR path
    b = ctx.classify(ds.query_off, ds.query_codes, eo, eids, taps=("counts", "hist", "kmers"))
    assert _same_outputs(a, b)
    assert np.array_equal(a.counts, b.counts) and np.array_equal(a.hist, b.hist) and np.array_equal(a.n_kmers, b.n_kmers)
    assert bytes_seq == ctx.index_bytes
    # reference shard of the same tree: rows restricted to the k-mers present in the shard, either way
    N = ht.num_tips
    outs = []
    for t in (capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes), ht):
        ctx.upload_tree(t, (N // 3, 2 * N // 3))
        outs.append(ctx.classify(ds.query_off, ds.query_codes, eo, eids, taps=("counts", "hist")))
    assert np.array_equal(outs[0].counts, outs[1].counts) and np.array_equal(outs[0].hist, outs[1].hist)
    assert np.array_equal(outs[0].counts, a.counts[:, N // 3: 2 * N // 3])


def test_pipelined_batch_matches_serial(ctx):
    """A batch large enough for the two-stream sub-batch pipeline (>= 4096 queries) must give bit-identical outputs with the
    pipeline on (default), off, and with an odd sub-batch size; taps included."""
    ds = synth.generate("small", n_queries=4500, measure=False)
    ht = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes)
    ctx.upload_tree(ht)
    eo, eids = ht.exact_batch(ds.query_off, ds.query_codes)
    outs = []
    try:
        for pipe, sb in ((1, 0), (0, 0), (1, 777)):
            ctx.set_option(capi.RTX_OPT_PIPELINE, pipe)
            ctx.set_option(capi.RTX_OPT_SUB_BATCH, sb)
            outs.append(ctx.classify(ds.query_off, ds.query_codes, eo, eids, taps=("counts", "hist", "probs")))
            if pipe and sb == 0:
                assert ctx.sub_batch < ds.n_queries  # really pipelined
    finally:
        ctx.set_option(capi.RTX_OPT_PIPELINE, 1)
        ctx.set_option(capi.RTX_OPT_SUB_BATCH, 0)
    for o in outs[1:]:
        assert _same_outputs(outs[0], o)
        assert np.array_equal(outs[0].counts, o.counts) and np.array_equal(outs[0].hist, o.hist)
        cnt = o.counts.astype(np.int64)
        assert np.array_equal(np.take_along_axis(outs[0].probs, cnt, 1), np.take_along_axis(o.probs, cnt, 1))  # P(m) where the histogram is non-zero


def test_16s_like_long_queries(oracle, ctx):
    ds = synth.generate("x16s", n_refs=1500, n_queries=48, length=1500, kind="16s", seed=77, measure=False)
    o, dev, ot, _ = _run_both(oracle, ctx, ds, skip=True)
    assert int(o["K"].max()) > 1023  # needs the 11-plane kernel
    _assert_integer_parity(o, dev, ds.n_queries)
    _assert_result_parity(o, dev, ot, ds.n_queries)


# ---- real data: golden sample of the reference's example file, used as its own database (SURVEY 8c) -------------------
def test_diptera_sample_self_classification(oracle, ctx):
    text = open(os.path.join(GOLDEN, "diptera_sample.fasta")).read()
    ot = oracle.Tree.from_fasta(text)
    ht = capi.Tree.from_fasta(text)
    labels, q_off, q_codes = oracle.parse_queries(text)
    ctx.upload_tree(ht)
    for skip in (False, True):
        eo, eids = ht.exact_batch(q_off, q_codes)
        dev = ctx.classify(q_off, q_codes, eo, eids, skip_exact=skip, taps=("counts", "hist", "kmers"))
        o = ot.classify(q_off, q_codes, skip_exact=skip, threads=4, chunk_size=16, want_counts=True, want_probs=True, want_kmers=True)
        _assert_integer_parity(o, dev, len(labels))
        _assert_result_parity(o, dev, ot, len(labels))
        golden = os.path.join(GOLDEN, "diptera_sample.skip.out" if skip else "diptera_sample.default.out")
        qs = capi.Queries.from_fasta(text)
        sent, _, _ = capi.raxtax(ctx, qs, ht, skip_exact_matches=skip)
        # every query whose lines differ from the golden text must be a documented tie / rounding-boundary case (tests/parity.py)
        parity.assert_text_parity([s[1].split("\n") for s in sent], parity.lines_by_query(open(golden).read(), labels), o, ot,
                                  what=f"diptera sample vs golden ({'skip' if skip else 'default'})")


# ---- edge cases ---------------------------------------------------------------------------------------------------------
def test_edge_cases(oracle, ctx):
    rng = np.random.default_rng(5)
    base = synth.BASE_CODES[rng.integers(0, 4, 120)]
    refs = [base.copy() for _ in range(6)]
    refs[1][50] = synth.BASE_CODES[(int(np.log2(refs[1][50])) + 1) % 4]
    refs[2] = synth.BASE_CODES[rng.integers(0, 4, 120)]
    refs[3] = base[:7]  # shorter than one 8-mer: no postings at all
    refs[4] = np.full(40, 15, np.uint8)  # all N
    refs[5] = base.copy()  # exact duplicate of ref 0 under another species
    lineages = ["k,p,a,s1", "k,p,a,s2", "k,q,b,s3", "k,q,b,s4", "k,q,c,s5", "k,r,d,s6"]
    queries = [base, base[:30], base[:8], base[:7], np.zeros(0, np.uint8), np.full(33, 15, np.uint8),
               synth.BASE_CODES[rng.integers(0, 4, 64)], refs[1], refs[2][10:90], np.full(20, 1, np.uint8)]
    r_off, r_codes = _pack(oracle, refs)
    q_off, q_codes = _pack(oracle, queries)
    for skip, raw in [(False, False), (True, False), (False, True)]:
        o, dev, ot, _ = _run_both(oracle, ctx, (lineages, r_off, r_codes, q_off, q_codes), skip=skip, raw=raw)
        _assert_integer_parity(o, dev, len(queries))
        _assert_result_parity(o, dev, ot, len(queries), max_tolerated_frac=1.0)
    # single-reference database
    o, dev, ot, _ = _run_both(oracle, ctx, (["only,one"], *_pack(oracle, [base]), q_off, q_codes))
    _assert_integer_parity(o, dev, len(queries))
    _assert_result_parity(o, dev, ot, len(queries), max_tolerated_frac=1.0)
    # empty batch
    dev = ctx.classify(np.zeros(1, np.uint64), np.zeros(0, np.uint8))
    assert len(dev.first_ref) == 0


def test_errors_are_loud(ctx):
    c2 = capi.Context(0)
    with pytest.raises(capi.RtxError) as ei:
        c2.classify(np.array([0, 8], np.uint64), np.ones(8, np.uint8))
    assert ei.value.code == capi.RTX_ERR_NO_INDEX
    c2.close()
    with pytest.raises(capi.RtxError):
        ctx.upload_index_arrays(0, np.zeros(65537, np.uint64), np.zeros(1, np.uint32), [0], [0], [0], [0], [0], [1])
    # options 5 and 8 are not assigned, walk variant 2 does not exist, a CTA holds at most 16 queries
    for opt, value in [(5, 0), (8, 0), (capi.RTX_OPT_WALK_VARIANT, 2), (capi.RTX_OPT_HITCOUNT_GROUP, 101)]:
        with pytest.raises(capi.RtxError) as ei:
            ctx.set_option(opt, value)
        assert ei.value.code == capi.RTX_ERR_INVALID


# ---- full-size properties (BASELINE configs 2, 3, 4 at their full reference counts, reduced query counts) -----------------------
def _check_scale_properties(ctx, ds, skip):
    """Size-independent properties of one classified batch: k-mer lists, histogram mass, the postings checksum
    sum_r count[r] == sum_k |postings(k)| (bit-exact, integer), result ordering, override / skip-exact handling."""
    ht = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes)
    ctx.upload_tree(ht)
    eo, eids = ht.exact_batch(ds.query_off, ds.query_codes)
    dev = ctx.classify(ds.query_off, ds.query_codes, eo, eids, skip_exact=skip, taps=("counts", "hist", "kmers"))
    N = ht.num_tips
    off, ids = ht.csr()
    lens = (off[1:] - off[:-1]).astype(np.int64)
    lin = ht.lineages
    n_override = 0
    for q in range(ds.n_queries):
        K = int(dev.n_kmers[q])
        km = dev.kmers[q, :K]
        assert np.array_equal(km, synth.kmers_of(ds.query_seq(q)))
        h = dev.hist[q, : K + 1].astype(np.int64)
        assert h.sum() == N  # every reference lands in exactly one bin
        ex = eids[eo[q]: eo[q + 1]].astype(np.int64)
        cnt = dev.counts[q].astype(np.int64)
        zeroed = int(K * len(ex)) if skip else 0  # an exact copy shares every k-mer; --skip-exact-matches zeroes it (raxtax.rs:65-68)
        assert (h * np.arange(K + 1)).sum() == cnt.sum() == lens[km.astype(np.int64)].sum() - zeroed  # checksum of postings
        assert np.array_equal(np.bincount(cnt, minlength=K + 1)[: K + 1], h)
        res = dev.for_query(q)
        assert res, "no empty result (raxtax.rs:72)"
        for fr, conf, local, glob in res:
            assert len(conf) == lin[fr].count(",") + 1
            assert np.all(np.diff(conf) <= 1e-12) and 0.0 < conf[-1] <= conf[0] <= 1.0 + 1e-12  # confidences shrink down the lineage
            assert 0.0 <= glob <= 1.0 and local >= 0.0
        confs = [tuple(c) for _, c, _, _ in res]
        assert confs == sorted(confs, reverse=True)  # lineage.rs:93
        if len(ex) == 1 and not skip:  # override (raxtax.rs:73-84)
            assert len(res) == 1 and res[0][0] == int(ex[0]) and np.all(res[0][1] == 1.0)
            n_override += 1
        if len(ex) >= 1:
            assert np.all(cnt[ex] == (0 if skip else K))
    return ht, eo, eids, dev, n_override


def test_c2_scale_properties(ctx):
    ds = synth.generate("c2", n_queries=300, measure=False)
    _, _, _, _, n_override = _check_scale_properties(ctx, ds, skip=False)
    assert n_override > 0


@pytest.mark.parametrize("cfg,nq,skip", [("c3", 256, False), ("c4", 256, True)])
def test_full_scale_configs(oracle, ctx, cfg, nq, skip):
    """BASELINE configs 3 (1 M COI refs) and 4 (500 k 16S-like 1500 bp refs, --skip-exact-matches) at their full reference
    counts: size-independent properties of every query, then full parity of all 256 queries against the CPU oracle built over
    the same references, on all host cores (RTX_FULL_ORACLE=0 skips the oracle part; it costs ~1-2 min of host time per config)."""
    ds = synth.generate(cfg, n_queries=nq, measure=False)
    ht, eo, eids, dev, _ = _check_scale_properties(ctx, ds, skip=skip)
    assert ht.num_tips == synth.CONFIGS[cfg][0]
    if os.environ.get("RTX_FULL_ORACLE", "1") != "0":
        n = nq
        ot = parity.oracle_tree_from_ds(oracle, ds)
        q_off = ds.query_off[: n + 1]
        q_codes = ds.query_codes[: int(q_off[-1])]
        o = ot.classify(q_off, q_codes, skip_exact=skip, threads=os.cpu_count() or 4, chunk_size=4, want_counts=True, want_probs=True, want_kmers=True)
        assert np.array_equal(o["K"], dev.n_kmers[:n])
        assert np.array_equal(o["counts"], dev.counts[:n]), "hit counts at full scale"
        checker = parity.TolerantChecker(ot.flatten(), ot.num_tips)
        ok, tol, bad = parity.compare_batch(o, dev, n, checker, o["probs"])
        assert not bad, f"{len(bad)} queries differ from the oracle at full scale, first {bad[:3]}"
        assert tol <= max(1, n // 20)
        print(f"{cfg}: {ok} of {n} queries identical to the oracle at N = {ht.num_tips}, {tol} within tie/rounding tolerance")


# ---- reference-sharded mode: several shards on ONE GPU (one context per shard), exchanges by device copies -----------------
@pytest.mark.parametrize("n_shards,skip,raw", [(2, False, False), (3, True, False), (5, False, True), (8, False, False)])  # 8 = BASELINE config 5's shard count
def test_reference_sharded_matches_oracle(oracle, n_shards, skip, raw):
    from raxtax_b200 import dist as rdist

    ds = synth.generate("small", n_queries=96, measure=False)
    seqs = [ds.ref_seq(i) for i in range(ds.n_refs)]
    ot = oracle.Tree.new(ds.ref_lineages, seqs)
    ht = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes)
    cuts = rdist.shard_cuts(ht.num_tips, n_shards)
    ctxs = [capi.Context(0) for _ in range(n_shards)]
    try:
        for r, c in enumerate(ctxs):
            c.upload_tree_sharded(ht, n_shards, r, cuts)
        eo, eids = ht.exact_batch(ds.query_off, ds.query_codes)
        ref_levels = ht.index_arrays()["ref_levels"]
        merged, outs = rdist.classify_sharded_local(ctxs, ds.query_off, ds.query_codes, eo, eids, ref_levels, skip_exact=skip, raw_conf=raw,
                                                    taps=("counts", "hist", "kmers"))
        o = ot.classify(ds.query_off, ds.query_codes, skip_exact=skip, raw_conf=raw, threads=4, chunk_size=16, want_counts=True, want_probs=True,
                        want_kmers=True)
        # integer parity: the shards' count vectors concatenate to the oracle's, the all-reduced histograms are the global ones
        assert np.array_equal(np.concatenate([x.counts for x in outs], axis=1), o["counts"])
        for q in range(ds.n_queries):
            K = int(o["K"][q])
            for x in outs:
                assert np.array_equal(parity.hist_from_counts(o["counts"][q], K), x.hist[q, : K + 1])
        assert np.array_equal(o["K"], merged.n_kmers)
        _assert_result_parity(o, merged, ot, ds.n_queries)
        # phases out of order are refused
        with pytest.raises(capi.RtxError):
            ctxs[0].shard_phase(3)
        with pytest.raises(capi.RtxError):
            ctxs[0].batch_run()
    finally:
        for c in ctxs:
            c.close()


# ---- the raxtax command-line binary (SURVEY 8f row 1): unchanged CLI flags and output files ---------------------------------
def test_cli_binary_writes_reference_format_files(oracle, tmp_path):
    import subprocess

    from raxtax_b200 import _build

    fasta = os.path.join(GOLDEN, "diptera_sample.fasta")
    for skip, golden in ((False, "diptera_sample.default.out"), (True, "diptera_sample.skip.out")):
        prefix = tmp_path / ("skip" if skip else "default")
        cmd = [_build.CLI_BIN, "-d", fasta, "-i", fasta, "-o", str(prefix), "--tsv", "--batch", "150"] + (["--skip-exact-matches"] if skip else [])
        r = subprocess.run(cmd, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        out = (prefix / "raxtax.out").read_text().split("\n")
        exp = open(os.path.join(GOLDEN, golden)).read().split("\n")
        assert len(out) == len(exp)
        text = open(fasta).read()
        ot = oracle.Tree.from_fasta(text)
        labels, q_off, q_codes = oracle.parse_queries(text)
        o = ot.classify(q_off, q_codes, skip_exact=skip, threads=4, chunk_size=16, want_probs=True)
        parity.assert_text_parity(parity.lines_by_query("\n".join(out), labels), parity.lines_by_query("\n".join(exp), labels), o, ot,
                                  what=f"CLI raxtax.out vs golden ({'skip' if skip else 'default'})")
        tsv = (prefix / "raxtax.tsv").read_text().split("\n")
        assert len(tsv) == len(exp) and tsv[0].count("\t") == 15  # label + 6 x (rank, conf) + 2 signals + sequence
        assert len((prefix / "raxtax.ckp").read_text().splitlines()) == 400
        log = (prefix / "raxtax.log").read_text()
        assert log.startswith("raxtax-b200") and ("Exact sequence match for query" in log) == (not skip)
        assert (prefix / "diptera_sample.bin").is_file() and (prefix / "raxtax.json").is_file()
        # a second run into the same folder continues from the checkpoint: every query is already processed, nothing is added
        r2 = subprocess.run(cmd, capture_output=True, text=True)
        assert r2.returncode == 0 and "Restarting from checkpoint" in r2.stderr
        assert (prefix / "raxtax.out").read_text().split("\n") == out


def test_cli_resumes_from_checkpoint_and_loads_bin(tmp_path):
    """io.rs:156-230: after an interruption (progress file short, a half-written result line in raxtax.out) the same command
    finishes the job from raxtax.json / raxtax.ckp with the database read back from the .bin, and the union equals one clean run."""
    import subprocess

    from raxtax_b200 import _build

    fasta = os.path.join(GOLDEN, "diptera_sample.fasta")
    clean, prefix = tmp_path / "clean", tmp_path / "resumed"
    base = [_build.CLI_BIN, "-d", fasta, "-i", fasta, "--tsv"]
    assert subprocess.run(base + ["-o", str(clean), "--skip-db"], capture_output=True, text=True).returncode == 0
    assert not list(clean.glob("*.bin"))  # --skip-db
    assert subprocess.run(base + ["-o", str(prefix)], capture_output=True, text=True).returncode == 0
    done = (prefix / "raxtax.ckp").read_text().splitlines()
    assert len(done) == 400
    keep = set(done[:137])
    (prefix / "raxtax.ckp").write_text("\n".join(done[:137]) + "\n")
    for name in ("raxtax.out", "raxtax.tsv"):  # results of unlisted queries stay behind, as after a kill between the two writes
        lines = (prefix / name).read_text().splitlines()
        cut = [l for l in lines if l.split("\t")[0] in keep] + [l for l in lines if l.split("\t")[0] == done[137]]
        (prefix / name).write_text("\n".join(cut) + "\n")
    r = subprocess.run(base + ["-o", str(prefix)], capture_output=True, text=True)
    assert r.returncode == 0 and "Restarting from checkpoint" in r.stderr, r.stderr
    assert sorted((prefix / "raxtax.ckp").read_text().splitlines()) == sorted(done)
    for name in ("raxtax.out", "raxtax.tsv"):
        assert sorted((prefix / name).read_text().splitlines()) == sorted((clean / name).read_text().splitlines()), name
    # --clean afterwards: checkpoint files and the database created under the prefix go, the user's -d file stays
    r = subprocess.run(base + ["-o", str(prefix), "--clean"], capture_output=True, text=True)
    assert r.returncode == 0
    assert not (prefix / "raxtax.json").exists() and not (prefix / "raxtax.ckp").exists() and not list(prefix.glob("*.bin"))
    assert os.path.exists(fasta)


def test_pinned_result_buffers_match_pageable(ctx):
    """rtx_host_alloc buffers (results written by DMA, ordered on the device) give exactly what ordinary memory gives."""
    ds = synth.generate("small", measure=False)
    ht = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes)
    ctx.upload_tree(ht)
    eo, eids = ht.exact_batch(ds.query_off, ds.query_codes)
    a = ctx.classify(ds.query_off, ds.query_codes, eo, eids)
    buf = ctx.pinned_results(ds.n_queries)
    for sub in (0, 37):  # one sub-batch, and several (results of different sub-batches interleave in the pool)
        ctx.set_option(capi.RTX_OPT_SUB_BATCH, sub)
        b = ctx.classify(ds.query_off, ds.query_codes, eo, eids, out=buf)
        ctx.set_option(capi.RTX_OPT_SUB_BATCH, 0)
        n = int(a.result_begin[-1])
        assert n > 0 and np.array_equal(a.result_begin, b.result_begin)
        assert np.array_equal(a.n_kmers, b.n_kmers) and np.array_equal(a.global_signal, b.global_signal)
        assert np.array_equal(a.first_ref, b.first_ref[:n]) and np.array_equal(a.n_levels, b.n_levels[:n])
        assert np.array_equal(a.confidence, b.confidence[:n]) and np.array_equal(a.local_signal, b.local_signal[:n])


def test_raxtax_multi_context_equals_single(ctx):
    """rxh_raxtax_multi (one host thread per context, chunks from a shared counter) sends exactly the lines rxh_raxtax sends;
    two contexts on the one GPU of the test box stand in for two GPUs."""
    ds = synth.generate("small", measure=False)
    ht = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes)
    qs = capi.Queries.new(ds.query_labels, ds.query_off, ds.query_codes)
    ctx.upload_tree(ht)
    one, logs1, warn1 = capi.raxtax(ctx, qs, ht, tsv=True)
    other = capi.Context(0)
    try:
        other.upload_tree(ht)
        two, logs2, warn2 = capi.raxtax([ctx, other], qs, ht, chunk_size=17, tsv=True)
    finally:
        other.close()
    assert [r[0] for r in one] == ds.query_labels  # single context: query order
    assert sorted(two) == sorted(one) and len(two) == len(one)
    assert sorted(logs1) == sorted(logs2) and warn1 == warn2


# ---- randomised differential test: odd tree shapes, ragged lengths, ambiguity codes, duplicates ----------------------------------
def _random_case(seed):
    rng = np.random.default_rng(1000 + seed)
    n_refs = int(rng.integers(1, 90))
    depth_max = int(rng.integers(1, 7))
    alphabet = ["a", "b", "c", "dd", "e"]
    lineages, refs = [], []
    root_seq = synth.BASE_CODES[rng.integers(0, 4, int(rng.integers(8, 260)))]
    for _ in range(n_refs):
        d = int(rng.integers(2, depth_max + 2))  # at least two ranks: raxtax.rs:49 unwraps the parent of the last rank
        lineages.append(",".join(alphabet[int(rng.integers(0, len(alphabet)))] for _ in range(d)))
        s = root_seq.copy()
        mut = rng.random(len(s)) < rng.choice([0.0, 0.02, 0.1, 0.5])
        s[mut] = synth.BASE_CODES[rng.integers(0, 4, int(mut.sum()))]
        if rng.random() < 0.2:
            s[rng.integers(0, len(s), 3)] = rng.choice([15, 5, 10, 3])  # N and two-fold IUPAC codes
        if rng.random() < 0.15:
            s = s[: int(rng.integers(0, len(s) + 1))]  # truncated, possibly shorter than one 8-mer or empty
        refs.append(s)
    queries = []
    for _ in range(int(rng.integers(1, 40))):
        r = rng.random()
        if r < 0.35:
            q = refs[int(rng.integers(0, n_refs))].copy()  # exact match (possibly of several references)
        elif r < 0.8:
            q = refs[int(rng.integers(0, n_refs))].copy()
            if len(q):
                mut = rng.random(len(q)) < 0.05
                q[mut] = synth.BASE_CODES[rng.integers(0, 4, int(mut.sum()))]
        else:
            q = synth.BASE_CODES[rng.integers(0, 4, int(rng.integers(0, 300)))]
        queries.append(q)
    return lineages, refs, queries


@pytest.mark.parametrize("seed", range(int(os.environ.get("RTX_FUZZ_SEEDS", "16"))))  # RTX_FUZZ_SEEDS=200 for a longer hunt
def test_random_shapes_against_oracle(oracle, ctx, seed):
    lineages, refs, queries = _random_case(seed)
    r_off, r_codes = _pack(oracle, refs)
    q_off, q_codes = _pack(oracle, queries)
    for skip, raw in [(False, False), (True, False), (False, True)]:
        o, dev, ot, ht = _run_both(oracle, ctx, (lineages, r_off, r_codes, q_off, q_codes), skip=skip, raw=raw, sub_batch=int(seed % 3) * 5)
        _assert_integer_parity(o, dev, len(queries))
        ok, tol = _assert_result_parity(o, dev, ot, len(queries), max_tolerated_frac=1.0)
        if tol == 0:  # the text the host driver sends (raxtax.out / raxtax.tsv lines, lineage.rs:17-48) against the oracle's formatting
            labels = [f"q{i} some read" for i in range(len(queries))]
            qs = capi.Queries.new(labels, q_off, q_codes)
            sent, _, _ = capi.raxtax(ctx, qs, ht, skip_exact_matches=skip, raw_confidence=raw, chunk_size=7, tsv=True)
            assert [x[0] for x in sent] == labels
            assert [l for x in sent for l in x[1].split("\n")] == oracle.format_results(ot, o["results"], labels).split("\n")
            assert [l for x in sent for l in x[2].split("\n")] == oracle.format_results(ot, o["results"], labels, q_off, q_codes, tsv=True).split("\n")


def test_context_reuse_across_indexes_of_different_depth(oracle, ctx):
    """One context, a shallow database then a deep one (then back): the result pool and its query-ordered copy are re-sized with
    max_levels; every run equals a fresh context's."""
    rng = np.random.default_rng(77)
    base = synth.BASE_CODES[rng.integers(0, 4, 150)]

    def db(depth, n):
        lin, refs = [], []
        for i in range(n):
            lin.append(",".join(f"r{l}_{(i >> (depth - 1 - l)) if l < depth - 1 else i}" for l in range(depth)))
            s = base.copy()
            mut = rng.random(len(s)) < 0.08
            s[mut] = synth.BASE_CODES[rng.integers(0, 4, int(mut.sum()))]
            refs.append(s)
        return lin, refs

    cases = [db(2, 40), db(9, 64), db(3, 24)]
    queries = [cases[1][1][5], cases[0][1][7], base, synth.BASE_CODES[rng.integers(0, 4, 90)]]
    q_off, q_codes = _pack(oracle, queries)
    for lin, refs in cases:
        r_off, r_codes = _pack(oracle, refs)
        ht = capi.Tree.new(lin, r_off, r_codes)
        eo, eids = ht.exact_batch(q_off, q_codes)
        ctx.upload_tree(ht)
        a = ctx.classify(q_off, q_codes, eo, eids)
        fresh = capi.Context(0)
        try:
            fresh.upload_tree(ht)
            b = fresh.classify(q_off, q_codes, eo, eids)
        finally:
            fresh.close()
        assert np.array_equal(a.result_begin, b.result_begin) and np.array_equal(a.first_ref, b.first_ref)
        assert np.array_equal(a.n_levels, b.n_levels) and np.array_equal(a.confidence, b.confidence)
        assert np.array_equal(a.local_signal, b.local_signal) and np.array_equal(a.global_signal, b.global_signal)
        assert a.confidence.shape[1] == max(l.count(",") + 1 for l in lin)


@pytest.mark.parametrize("seed", range(int(os.environ.get("RTX_FUZZ_SEEDS", "16")) // 2))
def test_random_shapes_walk_variants_and_shards(oracle, ctx, seed):
    """The same random cases through (i) the depth-first walker alone and the forced retry path -- bit-identical to the default
    level-synchronous walk -- and (ii) the reference-sharded phases with 2-4 shards cut at arbitrary references, against the oracle."""
    from raxtax_b200 import dist as rdist

    lineages, refs, queries = _random_case(5000 + seed)
    r_off, r_codes = _pack(oracle, refs)
    q_off, q_codes = _pack(oracle, queries)
    ht = capi.Tree.new(lineages, r_off, r_codes)
    eo, eids = ht.exact_batch(q_off, q_codes)
    skip = seed % 2 == 1
    ctx.upload_tree(ht)
    outs = []
    try:
        for variant, cap in ((0, 0), (1, 0), (0, 4), (3, 0), (4, 0)):  # 3 / 4: large-frontier paths of the level-synchronous walk off / forced
            ctx.set_option(capi.RTX_OPT_WALK_VARIANT, variant)
            ctx.set_option(capi.RTX_OPT_WALK_LOG_CAP, cap)
            outs.append(ctx.classify(q_off, q_codes, eo, eids, skip_exact=skip))
    finally:
        ctx.set_option(capi.RTX_OPT_WALK_VARIANT, 0)
        ctx.set_option(capi.RTX_OPT_WALK_LOG_CAP, 0)
    for o2 in outs[1:]:
        assert _same_outputs(outs[0], o2)
    n = ht.num_tips
    if n < 2:
        return
    rng = np.random.default_rng(seed)
    n_shards = int(min(n, rng.integers(2, 5)))
    cuts = np.concatenate([[0], np.sort(rng.choice(np.arange(1, n), n_shards - 1, replace=False)), [n]]).astype(np.uint64)
    ctxs = [capi.Context(0) for _ in range(n_shards)]
    try:
        for r, c in enumerate(ctxs):
            c.upload_tree_sharded(ht, n_shards, r, cuts)
            c.set_option(capi.RTX_OPT_WALK_VARIANT, (0, 4, 1)[seed % 3])  # sharded walk: default, large-frontier paths forced, depth-first only
        ref_levels = ht.index_arrays()["ref_levels"]
        merged, per_rank = rdist.classify_sharded_local(ctxs, q_off, q_codes, eo, eids, ref_levels, skip_exact=skip, taps=("counts",))
    finally:
        for c in ctxs:
            c.close()
    ot = oracle.Tree.new(lineages, [np.asarray(r, np.uint8) for r in refs])
    o = ot.classify(q_off, q_codes, skip_exact=skip, threads=2, chunk_size=8, want_counts=True, want_probs=True)
    assert np.array_equal(np.concatenate([x.counts for x in per_rank], axis=1), o["counts"])
    _assert_result_parity(o, merged, ot, len(queries), max_tolerated_frac=1.0)


def _random_case_mid(seed):
    """Mid-size random databases: several reference tiles and prefix segments with ragged tails, query lengths that land in every
    counter-plane instantiation of the hit-count kernel (K < 256 / 1024 / 2048 / 8192), clade-structured similarity."""
    rng = np.random.default_rng(9000 + seed)
    n_refs = int(rng.choice([97, 511, 513, 2047, 2049, 4097, 6000]) + rng.integers(0, 40))
    length = int(rng.choice([40, 200, 650, 1100, 2600]))
    depth = int(rng.integers(2, 7))
    fan = [int(rng.integers(1, 6)) for _ in range(depth)]
    root = synth.BASE_CODES[rng.integers(0, 4, length)]
    clade_seq = {(): root}
    lineages, refs = [], []
    for _ in range(n_refs):
        path = tuple(int(rng.integers(0, f)) for f in fan)
        for d in range(1, depth + 1):
            key = path[:d]
            if key not in clade_seq:
                s = clade_seq[key[:-1]].copy()
                mut = rng.random(length) < 0.04
                s[mut] = synth.BASE_CODES[rng.integers(0, 4, int(mut.sum()))]
                clade_seq[key] = s
        s = clade_seq[path].copy()
        mut = rng.random(length) < rng.choice([0.0, 0.01, 0.05])
        s[mut] = synth.BASE_CODES[rng.integers(0, 4, int(mut.sum()))]
        if rng.random() < 0.05:
            s[rng.integers(0, length, 4)] = 15
        if rng.random() < 0.05:
            s = s[: int(rng.integers(0, length + 1))]
        lineages.append(",".join(f"L{d}_{path[d]}" for d in range(depth)))
        refs.append(s)
    queries = []
    for _ in range(int(rng.integers(3, 70))):
        q = refs[int(rng.integers(0, n_refs))].copy()
        r = rng.random()
        if r > 0.3 and len(q):
            mut = rng.random(len(q)) < rng.choice([0.01, 0.08, 0.3])
            q[mut] = synth.BASE_CODES[rng.integers(0, 4, int(mut.sum()))]
        if r > 0.9:
            q = synth.BASE_CODES[rng.integers(0, 4, int(rng.integers(0, length + 50)))]
        queries.append(q)
    return lineages, refs, queries


@pytest.mark.parametrize("seed", range(max(2, int(os.environ.get("RTX_FUZZ_SEEDS", "16")) // 4)))
def test_random_mid_size_against_oracle(oracle, ctx, seed):
    lineages, refs, queries = _random_case_mid(seed)
    r_off, r_codes = _pack(oracle, refs)
    q_off, q_codes = _pack(oracle, queries)
    skip, variant = bool(seed & 1), (capi.RTX_HITCOUNT_CSR if seed % 5 == 4 else capi.RTX_HITCOUNT_BITROWS)
    ctx.set_option(capi.RTX_OPT_WALK_VARIANT, 4 if seed % 3 == 1 else 0)  # every third case: the walk's large-frontier paths forced
    try:
        o, dev, ot, _ = _run_both(oracle, ctx, (lineages, r_off, r_codes, q_off, q_codes), skip=skip, sub_batch=int(seed % 4) * 7, variant=variant)
    finally:
        ctx.set_option(capi.RTX_OPT_WALK_VARIANT, 0)
    _assert_integer_parity(o, dev, len(queries))
    _assert_result_parity(o, dev, ot, len(queries), max_tolerated_frac=1.0)


@pytest.mark.parametrize("n_shards,skip", [(1, False), (3, False), (4, True)])
def test_giant_nodes_walk_paths(oracle, ctx, n_shards, skip):
    """A taxonomy with giant nodes (one genus holding thousands of species, one family holding hundreds of genera), so that the
    level-synchronous walk takes its large-frontier paths at their production thresholds -- mass-pruned search for significant
    children, fallback arg-max over the kept segments / in one pass -- unsharded (against the dense expansion, the depth-first
    walker and the oracle) and reference-sharded with cuts inside the giant nodes (against the oracle)."""
    from raxtax_b200 import dist as rdist

    rng = np.random.default_rng(77)
    L = 120
    root = synth.BASE_CODES[rng.integers(0, 4, L)]

    def mutate(s, rate):
        t = s.copy()
        m = rng.random(L) < rate
        t[m] = synth.BASE_CODES[rng.integers(0, 4, int(m.sum()))]
        return t

    lineages, refs = [], []
    fam_seq = [mutate(root, 0.15) for _ in range(3)]
    for f in range(3):
        n_gen = (900, 3, 1)[f]
        for g in range(n_gen):
            gs = mutate(fam_seq[f], 0.08)
            n_spe = 3000 if (f == 1 and g == 0) else (1200 if (f == 0 and g == 7) else int(rng.integers(1, 4)))
            for sp in range(n_spe):
                ss = mutate(gs, 0.05)
                for _ in range(int(rng.integers(1, 3))):
                    lineages.append(f"p:P,f:F{f},g:G{f}_{g},s:S{f}_{g}_{sp}")
                    refs.append(mutate(ss, 0.01))
    order = rng.permutation(len(refs))
    lineages = [lineages[i] for i in order]
    refs = [refs[i] for i in order]
    queries = []
    for _ in range(120):
        r = rng.random()
        base = refs[int(rng.integers(0, len(refs)))]
        if r < 0.3:
            queries.append(base.copy())
        elif r < 0.6:
            queries.append(mutate(base, 0.02))
        elif r < 0.85:
            queries.append(mutate(base, 0.25))  # flat profiles: fallback chains through the giant nodes
        else:
            queries.append(synth.BASE_CODES[rng.integers(0, 4, int(rng.integers(0, L)))])
    r_off, r_codes = _pack(oracle, refs)
    q_off, q_codes = _pack(oracle, queries)
    ht = capi.Tree.new(lineages, r_off, r_codes)
    eo, eids = ht.exact_batch(q_off, q_codes)
    ot = oracle.Tree.new(lineages, [np.asarray(r, np.uint8) for r in refs])
    o = ot.classify(q_off, q_codes, skip_exact=skip, threads=os.cpu_count() or 4, chunk_size=8, want_counts=True, want_probs=True)
    if n_shards == 1:
        ctx.upload_tree(ht)
        outs = []
        try:
            for variant in (0, 3, 1, 4):
                ctx.set_option(capi.RTX_OPT_WALK_VARIANT, variant)
                outs.append(ctx.classify(q_off, q_codes, eo, eids, skip_exact=skip, taps=("counts",)))
        finally:
            ctx.set_option(capi.RTX_OPT_WALK_VARIANT, 0)
        for o2 in outs[1:]:
            assert _same_outputs(outs[0], o2)
        assert np.array_equal(outs[0].counts, o["counts"])
        _assert_result_parity(o, outs[0], ot, len(queries), max_tolerated_frac=1.0)
        return
    n = ht.num_tips
    cuts = np.array([0] + [int(n * (i + 0.37) / n_shards) for i in range(n_shards - 1)] + [n], np.uint64)
    ref_levels = ht.index_arrays()["ref_levels"]
    for variant in (0, 1):
        ctxs = [capi.Context(0) for _ in range(n_shards)]
        try:
            for r, c in enumerate(ctxs):
                c.upload_tree_sharded(ht, n_shards, r, cuts)
                c.set_option(capi.RTX_OPT_WALK_VARIANT, variant)
            merged, per_rank = rdist.classify_sharded_local(ctxs, q_off, q_codes, eo, eids, ref_levels, skip_exact=skip, taps=("counts",))
        finally:
            for c in ctxs:
                c.close()
        assert np.array_equal(np.concatenate([x.counts for x in per_rank], axis=1), o["counts"])
        _assert_result_parity(o, merged, ot, len(queries), max_tolerated_frac=1.0)


def test_host_driver_dedups_identical_queries(ctx):
    """rxh_raxtax classifies every distinct sequence of a chunk once; the lines sent per query label (and the exact-match log lines)
    are those of the plain one-by-one path (RXH_NO_DEDUP=1)."""
    ds = synth.generate("small", n_queries=60, measure=False)
    rng = np.random.default_rng(4)
    pick = rng.integers(0, 60, 200)  # 200 queries drawn from 60 distinct sequences
    seqs = [ds.query_seq(int(i)) for i in pick]
    off = np.zeros(len(seqs) + 1, np.uint64)
    off[1:] = np.cumsum([len(s) for s in seqs])
    qs = capi.Queries.new([f"read{j}_{int(i)}" for j, i in enumerate(pick)], off, np.concatenate(seqs))
    ht = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes)
    ctx.upload_tree(ht)
    ctx.profile_reset()
    a = capi.raxtax(ctx, qs, ht, chunk_size=64, tsv=True)
    n_dedup = ctx.profile()["queries"]
    os.environ["RXH_NO_DEDUP"] = "1"
    try:
        ctx.profile_reset()
        b = capi.raxtax(ctx, qs, ht, chunk_size=64, tsv=True)
        n_plain = ctx.profile()["queries"]
    finally:
        del os.environ["RXH_NO_DEDUP"]
    assert a == b
    assert n_plain == 200 and n_dedup < 200  # the device saw fewer queries


@pytest.mark.parametrize("n_taxa", [190, 200, 201, 210, 256])
def test_many_equally_likely_taxa(oracle, ctx, n_taxa):
    """n identical references under n different species: every species gets 1/n.  n < 200 -> n result lines (1/n > 0.005 rounds to
    0.01; 200 is the most lines a query can produce), n > 200 -> nothing is significant below the genus and the fallback takes one of
    n exactly tied children (lineage.rs:156-164: which one is ulp noise in the reference, the checker accepts any of the tied)."""
    rng = np.random.default_rng(11)
    seq = synth.BASE_CODES[rng.integers(0, 4, 120)]
    other = synth.BASE_CODES[rng.integers(0, 4, 120)]
    lineages = [f"k,g,s{i:03d}" for i in range(n_taxa)] + ["k,h,x"]
    refs = [seq.copy() for _ in range(n_taxa)] + [other]
    r_off, r_codes = _pack(oracle, refs)
    q_off, q_codes = _pack(oracle, [seq, seq[:60], other])
    for skip, raw in [(False, False), (False, True), (True, False)]:
        o, dev, ot, _ = _run_both(oracle, ctx, (lineages, r_off, r_codes, q_off, q_codes), skip=skip, raw=raw)
        _assert_integer_parity(o, dev, 3)
        _assert_result_parity(o, dev, ot, 3, max_tolerated_frac=1.0)
        if not skip and n_taxa != 200:  # 1/200 sits exactly on the rounding boundary: the reference itself reports 190 of the 200
            n_lines = int(dev.result_begin[1] - dev.result_begin[0])
            assert n_lines == (n_taxa if n_taxa < 200 else 1), n_lines


def test_documented_limits(oracle, ctx):
    """The envelope INTEGRATION.md states: lineages of up to RTX_MAX_LEVELS = 32 ranks (one more is refused loudly, never mis-computed),
    queries of any length raxtax.rs:56 admits as far as the probability scratch fits device memory (tables in shared memory up to
    ~6.4 kb, in global scratch beyond)."""
    rng = np.random.default_rng(21)
    base = synth.BASE_CODES[rng.integers(0, 4, 300)]

    def db(depth):
        lin, refs = [], []
        for i in range(12):
            lin.append(",".join(f"r{l}_{i if l >= depth - 2 else 0}" for l in range(depth)))
            s = base.copy()
            mut = rng.random(len(s)) < 0.05 * (i % 4)
            s[mut] = synth.BASE_CODES[rng.integers(0, 4, int(mut.sum()))]
            refs.append(s)
        return lin, refs

    lin, refs = db(32)
    q_off, q_codes = _pack(oracle, [refs[3], base, base[:100]])
    o, dev, ot, _ = _run_both(oracle, ctx, (lin, *_pack(oracle, refs), q_off, q_codes))
    _assert_integer_parity(o, dev, 3)
    _assert_result_parity(o, dev, ot, 3, max_tolerated_frac=1.0)
    assert dev.confidence.shape[1] == 32
    assert ctx.hitcount_kernel_name().startswith("hitcount_bitrows_kernel<")  # fewer queries than a query group: the single-query kernel
    lin33, refs33 = db(33)
    with pytest.raises(capi.RtxError) as ei:
        ctx.upload_tree(capi.Tree.new(lin33, *_pack(oracle, refs33)))
    assert ei.value.code == capi.RTX_ERR_UNSUPPORTED
    # long queries: 6.3 kb (about 6 300 unique 8-mers) against 6.3 kb references
    long_base = synth.BASE_CODES[rng.integers(0, 4, 6300)]
    lrefs = []
    for i in range(20):
        s = long_base.copy()
        mut = rng.random(len(s)) < 0.02 * (i % 5)
        s[mut] = synth.BASE_CODES[rng.integers(0, 4, int(mut.sum()))]
        lrefs.append(s)
    llin = [f"k,p{i % 2},g{i % 5},s{i}" for i in range(20)]
    lq = [lrefs[7], long_base[100:6250], long_base[:900]]
    o, dev, ot, _ = _run_both(oracle, ctx, (llin, *_pack(oracle, lrefs), *_pack(oracle, lq)))
    _assert_integer_parity(o, dev, 3)
    _assert_result_parity(o, dev, ot, 3, max_tolerated_frac=1.0)
    assert int(dev.n_kmers.max()) > 5500
    # beyond ~6.4 kb the per-query tables of the probability kernel move to global scratch: 9 kb and 21 kb queries (a mitochondrial
    # genome) against references of that length
    for length in (9000, 21000):
        gbase = synth.BASE_CODES[rng.integers(0, 4, length)]
        grefs = []
        for i in range(10):
            s = gbase.copy()
            mut = rng.random(len(s)) < 0.01 * (i % 4)
            s[mut] = synth.BASE_CODES[rng.integers(0, 4, int(mut.sum()))]
            grefs.append(s)
        glin = [f"k,p{i % 2},g{i % 3},s{i}" for i in range(10)]
        gq = [grefs[3], gbase[50:length - 70], gbase[:700]]
        o, dev, ot, _ = _run_both(oracle, ctx, (glin, *_pack(oracle, grefs), *_pack(oracle, gq)), skip=length == 21000)
        _assert_integer_parity(o, dev, 3)
        _assert_result_parity(o, dev, ot, 3, max_tolerated_frac=1.0)
        assert int(dev.n_kmers.max()) > length * 0.85
        if length == 21000:  # row list and histogram too large for a warp's shared memory: the single-query kernel
            assert ctx.hitcount_kernel_name().startswith("hitcount_bitrows_kernel<")
    # raxtax.rs:56 asserts at most 65 535 unique 8-mers; longer queries are refused, loudly
    with pytest.raises(capi.RtxError) as ei:
        ctx.classify(*_pack(oracle, [synth.BASE_CODES[rng.integers(0, 4, 70000)]]))
    assert ei.value.code == capi.RTX_ERR_UNSUPPORTED


@pytest.mark.parametrize("n_shards,skip", [(3, False), (2, True)])
def test_host_driver_sharded_equals_unsharded(ctx, n_shards, skip):
    """rxh_raxtax_sharded (all shards driven by one process: phases + the in-process histogram / record exchanges + the merge) sends the
    lines rxh_raxtax sends for the unsharded index; contexts on the one GPU of the test box stand in for several GPUs."""
    from raxtax_b200 import dist as rdist

    ds = synth.generate("small", n_queries=150, measure=False)
    ht = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes)
    qs = capi.Queries.new(ds.query_labels, ds.query_off, ds.query_codes)
    ctx.upload_tree(ht)
    one, logs1, warn1 = capi.raxtax(ctx, qs, ht, skip_exact_matches=skip, tsv=True)
    cuts = rdist.shard_cuts(ht.num_tips, n_shards)
    shards = [capi.Context(0) for _ in range(n_shards)]
    try:
        for r, c in enumerate(shards):
            c.upload_tree_sharded(ht, n_shards, r, cuts)
        many, logs2, warn2 = capi.raxtax(shards, qs, ht, skip_exact_matches=skip, chunk_size=64, tsv=True, sharded=True)
    finally:
        for c in shards:
            c.close()
    assert [x[0] for x in many] == ds.query_labels
    same = sum(a == b for a, b in zip(one, many))
    assert same >= len(one) - 2, [(a, b) for a, b in zip(one, many) if a != b][:2]  # ulp-level ties may fall differently per shard sum
    assert sorted(logs1) == sorted(logs2) and warn1 == warn2
