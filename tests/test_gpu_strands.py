"""--strand both on the GPU (RTX_BOTH_STRANDS): the orientation the device picks follows the rule M(rc(s)) > M(s) computed from the
oracle's counts of both orientations, and everything the device reports for a query is the oracle's classification of the chosen
orientation -- through every path the batch can take."""
import ctypes as C
import os
import subprocess
from collections import Counter

import numpy as np
import pytest

from raxtax_b200 import capi, synth
from tests.test_gpu_parity import _assert_integer_parity, _assert_result_parity, _same_outputs

pytestmark = pytest.mark.gpu
TAPS = ("counts", "hist", "kmers", "probs")


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


def _pack(seqs):
    off = np.zeros(len(seqs) + 1, np.uint64)
    off[1:] = np.cumsum([len(s) for s in seqs])
    codes = np.concatenate([np.asarray(s, np.uint8) for s in seqs]) if seqs else np.zeros(0, np.uint8)
    return off, codes


def _mixed_set(long_query=False):
    """The tiny synthetic set with about half of the queries reverse-complemented, plus a palindrome, a read without a single
    unambiguous 8-mer (K = 0), a query that is the reverse complement of a reference and -- optionally -- a 7.5 kb query (the
    probability tables of such a query live in global scratch)."""
    ds = synth.generate("tiny", measure=False)
    flip = np.random.default_rng(1234).random(ds.n_queries) < 0.5
    codes = synth.reverse_complement_batch(ds.query_off, ds.query_codes, flip)
    seqs = [codes[int(ds.query_off[i]): int(ds.query_off[i + 1])] for i in range(ds.n_queries)]
    half = ds.ref_seq(7)[:120]
    seqs.append(np.concatenate([half, synth.reverse_complement(half)]))  # palindrome: both strands have the same 8-mers
    seqs.append(np.full(40, 15, np.uint8))  # all N: K = 0
    seqs.append(synth.reverse_complement(ds.ref_seq(11)))
    if long_query:
        seqs.append(synth.reverse_complement(np.concatenate([ds.ref_seq(i) for i in range(40, 65)])))
    off, codes = _pack(seqs)
    return ds, off, codes


def _oracle_expectation(oracle, ds, q_off, q_codes, skip, raw):
    """-> (rule strand per query, oracle output on the chosen orientations, oracle tree)"""
    ot = oracle.Tree.new(ds.ref_lineages, [ds.ref_seq(i) for i in range(ds.n_refs)])
    kw = dict(skip_exact=skip, raw_conf=raw, threads=4, chunk_size=16, want_counts=True, want_probs=True, want_kmers=True)
    fwd = ot.classify(q_off, q_codes, **kw)
    rev = ot.classify(q_off, synth.reverse_complement_batch(q_off, q_codes), **kw)
    M = lambda o: o["counts"].max(axis=1) if o["counts"].shape[1] else np.zeros(len(q_off) - 1)
    rule = (M(rev) > M(fwd)).astype(np.uint8)
    assert np.array_equal(fwd["K"], rev["K"])  # n_kmers does not depend on the strand
    oriented = synth.reverse_complement_batch(q_off, q_codes, rule.astype(bool))
    return rule, ot.classify(q_off, oriented, **kw), ot


def _classify_both(ctx, ht, q_off, q_codes, skip, raw, taps=TAPS):
    eo, eids = ht.exact_batch_both_strands(q_off, q_codes)
    assert len(eo) == 2 * (len(q_off) - 1) + 1
    return ctx.classify(q_off, q_codes, eo, eids, skip_exact=skip, raw_conf=raw, taps=taps, both_strands=True)


@pytest.mark.parametrize("skip,raw", [(False, False), (True, False), (False, True)])
def test_both_strands_follow_rule_and_match_oracle(oracle, ctx, skip, raw):
    ds, q_off, q_codes = _mixed_set()
    nq = len(q_off) - 1
    rule, o, ot = _oracle_expectation(oracle, ds, q_off, q_codes, skip, raw)
    ht = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes)
    ctx.upload_tree(ht)
    dev = _classify_both(ctx, ht, q_off, q_codes, skip, raw)
    assert np.array_equal(dev.strand, rule), f"device strands differ from the rule at {np.nonzero(dev.strand != rule)[0][:10]}"
    assert 0.3 < rule[: ds.n_queries].mean() < 0.7  # the set really mixes orientations
    assert rule[ds.n_queries] == 0 and rule[ds.n_queries + 1] == 0  # palindrome and K = 0 read: ties stay forward
    if not skip:  # with --skip-exact-matches the reference it equals no longer counts
        assert rule[ds.n_queries + 2] == 1
    _assert_integer_parity(o, dev, nq)
    _assert_result_parity(o, dev, ot, nq)


@pytest.mark.parametrize("skip", [False, True])
def test_both_strands_every_path_identical(ctx, skip):
    ds, q_off, q_codes = _mixed_set()
    ht = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes)
    ctx.upload_tree(ht)
    ref = _classify_both(ctx, ht, q_off, q_codes, skip, False)
    outs = {}
    try:
        ctx.set_option(capi.RTX_OPT_SUB_BATCH, 7)
        outs["sub-batch 7"] = _classify_both(ctx, ht, q_off, q_codes, skip, False)
        ctx.set_option(capi.RTX_OPT_PIPELINE, 1)
        outs["pipelined"] = _classify_both(ctx, ht, q_off, q_codes, skip, False)
        ctx.set_option(capi.RTX_OPT_PIPELINE, 0)
        ctx.set_option(capi.RTX_OPT_SUB_BATCH, 0)
        ctx.set_option(capi.RTX_OPT_HITCOUNT_GROUP, 1)
        outs["single-query K2"] = _classify_both(ctx, ht, q_off, q_codes, skip, False)
        ctx.set_option(capi.RTX_OPT_HITCOUNT_GROUP, 0)
        # both batch slots in flight: slot 1 holds a plus-mode batch of the same queries
        eo, eids = ht.exact_batch_both_strands(q_off, q_codes)
        eo1, eids1 = ht.exact_batch(q_off, q_codes)
        ctx.batch_slot(0)
        ctx.batch_upload(q_off, q_codes, eo, eids, skip_exact=skip, both_strands=True)
        ctx.batch_run()
        ctx.batch_slot(1)
        ctx.batch_upload(q_off, q_codes, eo1, eids1, skip_exact=skip)
        ctx.batch_run()
        ctx.batch_slot(0)
        outs["slot 0 of two"] = ctx.batch_download(taps=("hist", "kmers"))
        ctx.batch_slot(1)
        plain = ctx.batch_download()
        assert plain.strand is None
        with pytest.raises(capi.RtxError) as ei:
            ctx.batch_strands(len(q_off) - 1)
        assert ei.value.code == capi.RTX_ERR_INVALID
        ctx.batch_slot(0)
        # the CSR postings instead of the bit rows
        ctx.set_option(capi.RTX_OPT_KEEP_CSR, 1)
        ctx.set_option(capi.RTX_OPT_HITCOUNT_VARIANT, capi.RTX_HITCOUNT_CSR)
        ht_csr = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes, eager_kmer_map=True)
        ctx.upload_tree(ht_csr)
        outs["CSR"] = _classify_both(ctx, ht_csr, q_off, q_codes, skip, False)
    finally:
        ctx.batch_slot(0)
        for opt, v in ((capi.RTX_OPT_SUB_BATCH, 0), (capi.RTX_OPT_PIPELINE, 0), (capi.RTX_OPT_HITCOUNT_GROUP, 0),
                       (capi.RTX_OPT_HITCOUNT_VARIANT, capi.RTX_HITCOUNT_BITROWS), (capi.RTX_OPT_KEEP_CSR, 0)):
            ctx.set_option(opt, v)
    for name, o in outs.items():
        assert _same_outputs(ref, o), name
        assert np.array_equal(ref.strand, o.strand), name
        if o.counts is not None:
            assert np.array_equal(ref.counts, o.counts) and np.array_equal(ref.hist, o.hist), name
        if o.hist is not None:
            assert np.array_equal(ref.hist, o.hist) and np.array_equal(ref.kmers, o.kmers), name


def test_both_strands_long_query(oracle, ctx):
    ds, q_off, q_codes = _mixed_set(long_query=True)
    nq = len(q_off) - 1
    assert int(q_off[-1] - q_off[-2]) > 6400
    rule, o, ot = _oracle_expectation(oracle, ds, q_off, q_codes, False, False)
    ht = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes)
    ctx.upload_tree(ht)
    dev = _classify_both(ctx, ht, q_off, q_codes, False, False)
    assert np.array_equal(dev.strand, rule) and rule[-1] == 1
    _assert_integer_parity(o, dev, nq)
    _assert_result_parity(o, dev, ot, nq)
    # the other queries are classified as without the long one
    short = _classify_both(ctx, ht, q_off[:-1], q_codes[: int(q_off[-2])], False, False, taps=())
    for q in range(nq - 1):
        a, b = dev.for_query(q), short.for_query(q)
        assert len(a) == len(b) and all(x[0] == y[0] and np.array_equal(x[1], y[1]) for x, y in zip(a, b)), q
    assert np.array_equal(dev.strand[:-1], short.strand)


def test_both_strands_refused_where_unsupported(ctx):
    ds, q_off, q_codes = _mixed_set()
    ht = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes)
    ctx.upload_tree(ht)
    eo, eids = ht.exact_batch_both_strands(q_off, q_codes)
    L = capi.device_lib()
    ctx.batch_upload(q_off, q_codes, eo, eids, both_strands=True)
    assert L.rtx_shard_phase1(ctx._h) == capi.RTX_ERR_UNSUPPORTED
    assert L.rtx_shard_run(ctx._h) == capi.RTX_ERR_UNSUPPORTED
    assert b"reference-sharded" in L.rtx_last_error(ctx._h)
    with pytest.raises(capi.RtxError) as ei:
        ctx.classify(q_off, q_codes, eo, eids, shard_root=0, both_strands=True)
    assert ei.value.code == capi.RTX_ERR_UNSUPPORTED
    # uploaded, not yet downloaded: no strands to report
    s = np.zeros(len(q_off) - 1, np.uint8)
    assert L.rtx_batch_strands(ctx._h, s.ctypes.data_as(C.POINTER(C.c_uint8))) == capi.RTX_ERR_INVALID
    # plus mode: no strands at all
    plain = ctx.classify(q_off, q_codes, *ht.exact_batch(q_off, q_codes))
    assert plain.strand is None
    assert L.rtx_batch_strands(ctx._h, s.ctypes.data_as(C.POINTER(C.c_uint8))) == capi.RTX_ERR_INVALID


# ---- the host driver and the CLI: --strand both on the committed diptera sample ---------------------------------------------------
GOLDEN_FASTA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "diptera_sample.fasta")


def _cli(*args):
    from raxtax_b200 import _build

    r = subprocess.run([_build.CLI_BIN, *map(str, args)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return r


def _lines(path):
    return [l for l in path.read_text().split("\n") if l]


@pytest.mark.parametrize("tsv,skip", [(False, False), (True, False), (False, True), (True, True)])
def test_cli_both_strands_equals_plain_run_on_oriented_file(ctx, tmp_path, tsv, skip):
    """raxtax --strand both on a file with a seeded subset of the queries reverse-complemented gives exactly what a plain run gives on
    the file in which every query reported `-` is replaced by its reverse complement -- lines (strand column removed) and exact-match
    log lines -- and the strand column is the device's rtx_batch_strands."""
    q = capi.Queries.from_fasta(open(GOLDEN_FASTA).read())
    labels = q.labels
    off, codes = q.arrays()
    flip = np.random.default_rng(77).random(len(labels)) < 0.4
    mixed = synth.reverse_complement_batch(off, codes, flip)
    (tmp_path / "mixed.fasta").write_text(synth._fasta(labels, off, mixed, 60))
    extra = ["--tsv"] if tsv else []
    extra += ["--skip-exact-matches"] if skip else []
    _cli("-d", GOLDEN_FASTA, "-i", tmp_path / "mixed.fasta", "-o", tmp_path / "both", "--skip-db", "--strand", "both", *extra)
    both = _lines(tmp_path / "both" / "raxtax.out")
    strand_of = {}
    for l in both:
        lab, s = l.split("\t", 1)[0], l.rsplit("\t", 1)[1]
        assert s in "+-" and strand_of.setdefault(lab, s) == s
    assert set(strand_of) == set(labels)
    minus = np.array([strand_of[l] == "-" for l in labels])
    if not skip:  # every query is a reference of the database: the flipped ones are found, the others stay as given
        assert minus[flip].all() and not minus[~flip].any()
    # the device's own decision on the same batch
    ht = capi.Tree.from_fasta(open(GOLDEN_FASTA).read())
    ctx.upload_tree(ht)
    eo, eids = ht.exact_batch_both_strands(off, mixed)
    dev = ctx.classify(off, mixed, eo, eids, skip_exact=skip, both_strands=True)
    assert np.array_equal(dev.strand.astype(bool), minus)
    # a plain run on the oriented file
    oriented = synth.reverse_complement_batch(off, mixed, minus)
    (tmp_path / "oriented.fasta").write_text(synth._fasta(labels, off, oriented, 60))
    _cli("-d", GOLDEN_FASTA, "-i", tmp_path / "oriented.fasta", "-o", tmp_path / "plain", "--skip-db", *extra)
    strip = lambda ls: [l.rsplit("\t", 1)[0] for l in ls]
    assert sorted(strip(both)) == sorted(_lines(tmp_path / "plain" / "raxtax.out"))
    if tsv:
        both_tsv = _lines(tmp_path / "both" / "raxtax.tsv")
        assert all(l.rsplit("\t", 1)[1] == strand_of[l.split("\t", 1)[0]] for l in both_tsv)
        assert sorted(strip(both_tsv)) == sorted(_lines(tmp_path / "plain" / "raxtax.tsv"))
    exact = lambda p: Counter(l for l in _lines(p / "raxtax.log") if "Exact" in l)
    assert exact(tmp_path / "both") == exact(tmp_path / "plain")
    if not skip:
        assert sum(exact(tmp_path / "both").values()) > 0
    # the Python driver: the same strings as the binary
    sent, logs, _ = capi.raxtax(ctx, capi.Queries.from_fasta((tmp_path / "mixed.fasta").read_text()), ht, skip_exact_matches=skip, tsv=tsv,
                                both_strands=True)
    assert sorted(l for s in sent for l in s[1].split("\n")) == sorted(both)
    assert Counter(m for lvl, m in logs if "Exact" in m) == Counter(l.split("] ", 1)[1] for l in exact(tmp_path / "both").elements())
