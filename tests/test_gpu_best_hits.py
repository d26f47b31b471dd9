"""Best hits on the GPU (RTX_OPT_BEST_HITS): each query's references with count >= 1, by count descending then id ascending, the
first min(T, #) of them, must equal the numpy selection over the query's final count row (tap_counts) bit for bit -- on synthetic
reads in every mode, through every path a batch can take, on exact-reference databases whose counts are laid out around the
threshold, segment and tile edges, with both strands, and through the host driver and the CLI.  Asking for them changes nothing
else a batch returns."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from raxtax_b200 import capi, synth
from tests import exact_reference as X
from tests.test_gpu_parity import _same_outputs

pytestmark = pytest.mark.gpu
TAPS = ("counts", "hist", "kmers", "probs")


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


def expected_hits(counts, T):
    """numpy reference: per row the ids with count >= 1 ordered by (count desc, id asc), the first T -> list of (ids, counts)."""
    out = []
    for row in np.asarray(counts):
        nz = np.nonzero(row)[0]
        sel = nz[np.lexsort((nz, -row[nz].astype(np.int64)))][:T]
        out.append((sel.astype(np.uint32), row[sel].astype(np.uint16)))
    return out


def assert_hits(dev, counts, T, what=""):
    n, ref, cnt = dev.best_hits
    assert ref.shape == (len(counts), T) and cnt.shape == (len(counts), T)
    for q, (ids, c) in enumerate(expected_hits(counts, T)):
        k = int(n[q])
        assert k == len(ids), f"{what} query {q}: {k} hits, expected {len(ids)}"
        assert np.array_equal(ref[q, :k], ids), f"{what} query {q}: ids {ref[q, :k][:12]} expected {ids[:12]}"
        assert np.array_equal(cnt[q, :k], c), f"{what} query {q}: counts"


def same_hits(a, b):
    (na, ra, ca), (nb, rb, cb) = a.best_hits, b.best_hits
    if not np.array_equal(na, nb):
        return False
    return all(np.array_equal(ra[q, :k], rb[q, :k]) and np.array_equal(ca[q, :k], cb[q, :k]) for q, k in enumerate(na))


def same_taps(a, b):
    return all(np.array_equal(getattr(a, t), getattr(b, t)) for t in TAPS if getattr(a, t) is not None)


def _pack(seqs):
    off = np.zeros(len(seqs) + 1, np.uint64)
    off[1:] = np.cumsum([len(s) for s in seqs])
    return off, np.concatenate([np.asarray(s, np.uint8) for s in seqs])


def _mixed_set(long_query=False):
    """200 reads of the small synthetic set (5 000 references: nine full 512-reference segments and a partial one), an all-N read
    (K = 0), an exact copy of a reference and -- optionally -- a 7.5 kb read (the global-scratch paths of the probability kernel
    and the single-query hit counting)."""
    ds = synth.generate("small", n_queries=200, measure=False)
    seqs = [ds.query_seq(i) for i in range(ds.n_queries)]
    seqs.append(np.full(40, 15, np.uint8))
    seqs.append(ds.ref_seq(4321).copy())
    if long_query:
        seqs.append(np.concatenate([ds.ref_seq(i) for i in range(40, 52)]))
    off, codes = _pack(seqs)
    return ds, off, codes


@pytest.fixture(scope="module")
def small(ctx):
    ds, off, codes = _mixed_set()
    ht = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes)
    return ds, ht, off, codes


def _classify(ctx, ht, off, codes, skip=False, raw=False, taps=TAPS, **kw):
    eo, eids = ht.exact_batch(off, codes)
    return ctx.classify(off, codes, eo, eids, skip_exact=skip, raw_conf=raw, taps=taps, **kw)


# ---- 1. synthetic reads: exact against numpy, nothing else changes ---------------------------------------------------------------
@pytest.mark.parametrize("skip,raw", [(False, False), (True, False), (False, True)])
def test_best_hits_match_numpy_and_change_nothing_else(ctx, small, skip, raw):
    ds, ht, off, codes = small
    ctx.upload_tree(ht)
    base = _classify(ctx, ht, off, codes, skip, raw)
    assert base.best_hits is None
    nq = len(off) - 1
    for T in (1, 10, 64):
        dev = _classify(ctx, ht, off, codes, skip, raw, best_hits=T)
        assert _same_outputs(base, dev) and same_taps(base, dev), T
        assert np.array_equal(base.n_kmers, dev.n_kmers)
        assert_hits(dev, dev.counts, T, f"T={T}")
        n = dev.best_hits[0]
        assert n[nq - 2] == 0  # K = 0
        assert n.max() == T  # the selection is full where enough references have hits
        if not skip:  # the exact copy of a reference leads its list with all K 8-mers shared
            assert dev.best_hits[2][nq - 1, 0] == dev.n_kmers[nq - 1]
    # T = 0 after T > 0: off again
    again = _classify(ctx, ht, off, codes, skip, raw)
    assert again.best_hits is None and _same_outputs(base, again)


# ---- 2. launch space: every path gives the same hits, and on every path the hits change nothing else ------------------------------
PATHS = [  # name, options set for the run (reset to the defaults afterwards), CSR postings kept in the index
    ("default", {}, False),
    *[(f"group {G}", {capi.RTX_OPT_HITCOUNT_GROUP: G}, False) for G in (1, 2, 4, 16)],
    ("sub-batch 8", {capi.RTX_OPT_SUB_BATCH: 8}, False),  # 202 / 203 queries: 25 full sub-batches and a partial one
    ("pipelined", {capi.RTX_OPT_SUB_BATCH: 8, capi.RTX_OPT_PIPELINE: 1}, False),
    ("CSR", {capi.RTX_OPT_HITCOUNT_VARIANT: capi.RTX_HITCOUNT_CSR}, True),
]
DEFAULTS = {capi.RTX_OPT_HITCOUNT_GROUP: 0, capi.RTX_OPT_SUB_BATCH: 0, capi.RTX_OPT_PIPELINE: 0,
            capi.RTX_OPT_HITCOUNT_VARIANT: capi.RTX_HITCOUNT_BITROWS, capi.RTX_OPT_KEEP_CSR: 0}


def test_best_hits_every_path_identical(ctx):
    """Two batches: the mixed set (result lines and signals are deterministic: they must not change with T), and the mixed set with
    a 7.5 kb read.  Such a read switches the probability kernel of the whole batch to one shared-memory sum array updated with
    atomics, whose summation order -- and so the last bits of the signals -- varies from run to run; that batch checks the hits
    (integers, fixed by the counts) and the counts only."""
    T = 10
    batches = {"mixed": _mixed_set(), "with 7.5 kb read": _mixed_set(long_query=True)}
    assert int(batches["with 7.5 kb read"][1][-1] - batches["with 7.5 kb read"][1][-2]) > 6400
    trees = {}
    ref = {}
    try:
        for name, opts, csr in PATHS:
            ctx.set_option(capi.RTX_OPT_KEEP_CSR, int(csr))
            for bname, (ds, off, codes) in batches.items():
                key = (bname, csr)
                if key not in trees:
                    trees[key] = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes, eager_kmer_map=csr)
                ht = trees[key]
                ctx.upload_tree(ht)
                for opt, v in opts.items():
                    ctx.set_option(opt, v)
                o = _classify(ctx, ht, off, codes, best_hits=T, taps=("counts",))
                deterministic = bname == "mixed"
                o0 = _classify(ctx, ht, off, codes, taps=()) if deterministic else None
                for opt in opts:
                    ctx.set_option(opt, DEFAULTS[opt])
                if name == "default":
                    assert_hits(o, o.counts, T, bname)
                    ref[bname] = (o0, o)
                    continue
                r0, r = ref[bname]
                assert np.array_equal(r.counts, o.counts), (name, bname)
                assert same_hits(r, o), (name, bname)
                if deterministic:
                    assert _same_outputs(r0, o0) and _same_outputs(o0, o), (name, bname)
        # upload / run / download on slot 0 while slot 1 holds another batch with T = 64
        ctx.set_option(capi.RTX_OPT_KEEP_CSR, 0)
        ds, off, codes = batches["mixed"]
        ht = trees[("mixed", False)]
        ctx.upload_tree(ht)
        eo, eids = ht.exact_batch(off, codes)
        ctx.batch_slot(0)
        ctx.batch_upload(off, codes, eo, eids, best_hits=T)
        ctx.batch_run()
        ctx.batch_slot(1)
        ctx.batch_upload(off[:51], codes[: int(off[50])], eo[:51], eids, best_hits=64)
        ctx.batch_run()
        ctx.batch_slot(0)
        mine = ctx.batch_download()
        ctx.batch_slot(1)
        other = ctx.batch_download(taps=("counts",))
        assert_hits(other, other.counts, 64, "slot 1")
        assert same_hits(ref["mixed"][1], mine) and _same_outputs(ref["mixed"][0], mine), "slot 0 of two"
    finally:
        ctx.batch_slot(0)
        for opt, v in DEFAULTS.items():
            ctx.set_option(opt, v)


# ---- 3. exact-reference databases: the selection's edge cases laid out on purpose --------------------------------------------------
N_EDGE = 1500  # not a multiple of 512: the last segment holds 476 references


def _edge_db():
    """References in construction order (the lineages sort that way).  Against the main read [5000, 5100) (K = 100): counts 95 at
    id N - 1 (last, partial segment) and 90 / 80 / 80 / 70 / 60 / 60 in segments 1 and 2, twelve ties at 50 spread over all three
    segments (T = 10 keeps the three lowest ids, all in segment 0, whose maximum is exactly 50), twenty references at 1..5, the
    rest 0.  The skip read [8000, 8080) has exact copies at ids 3 and 600 -- the only
    references of their segments above its threshold -- and a superstring at 1200."""
    rng = np.random.default_rng(2024)
    a, b = 5000, 5100
    wins = [None] * N_EDGE
    place = {N_EDGE - 1: 95, 700: 90, 1150: 80, 1100: 80, 513: 70, 1023: 60, 1024: 60}
    for pos in (1400, 200, 1450, 515, 90, 1030, 1498, 511, 800, 512, 10, 1300):
        place[pos] = 50
    for pos in rng.choice([p for p in range(512, N_EDGE) if p not in place and p not in (3, 600, 1200)], 20, replace=False):
        place[int(pos)] = int(rng.integers(1, 6))
    for pos, c in place.items():
        s = a + int(rng.integers(0, 100 - c + 1))
        wins[pos] = (s, s + c)
    wins[3] = wins[600] = (8000, 8080)
    wins[1200] = (7995, 8090)
    for pos in range(N_EDGE):
        if wins[pos] is None:
            s = int(rng.integers(20000, 30000))
            wins[pos] = (s, s + int(rng.integers(1, 24)))
    lineages = [f"root,g{j // 40:04d},r{j:05d}" for j in range(N_EDGE)]
    qs = [X.window_query(a, b, "main"), X.window_query(8000, 8080, "skip"), X.no_kmer_query(30, "all-N"),
          X.window_query(60000, 60050, "no shared 8-mer"), X.window_query(a + 40, a + 41, "K=1")]
    return X.ExactDb("best-hits edges", lineages, np.array(wins, np.int64), [X.window_seq(s, e) for s, e in wins], qs)


def _exact_run(ctx, db, T, skip=False, **kw):
    off, codes = db.packed_refs()
    ht = capi.Tree.new(db.lineages, off, codes)
    ctx.upload_tree(ht)
    qo, qc = db.packed_queries()
    eo, eids = ht.exact_batch(qo, qc)
    dev = ctx.classify(qo, qc, eo, eids, skip_exact=skip, taps=("counts",), best_hits=T, **kw)
    return dev, ht, eo, eids


def test_best_hits_exact_reference_edges(ctx):
    db = _edge_db()
    assert sorted(db.lineages) == db.lineages
    for T in (1, 10, 12, 64):
        dev, *_ = _exact_run(ctx, db, T)
        want = [db.counts(q) for q in db.queries]
        assert np.array_equal(dev.counts, np.array(want)), "closed-form counts"
        assert_hits(dev, want, T, f"T={T}")
    n, ref, cnt = _exact_run(ctx, db, 10)[0].best_hits
    # the tie run straddles the boundary: six above 50, then the four lowest ids of the twelve at 50
    assert list(ref[0, :10]) == [N_EDGE - 1, 700, 1100, 1150, 513, 1023, 1024, 10, 90, 200]
    assert list(cnt[0, :10]) == [95, 90, 80, 80, 70, 60, 60, 50, 50, 50]
    assert n[2] == 0 and n[3] == 0  # K = 0; no shared 8-mer
    # fewer than T references with a hit: all of them (39 for the main read, one row for the K = 1 read)
    n64 = _exact_run(ctx, db, 64)[0].best_hits[0]
    assert n64[0] == 39 and n64[4] == int((db.counts(db.queries[4]) > 0).sum())
    # the same with every path the hit counting can take; before each, a batch of as many all-N reads leaves per-segment maxima of 0
    # in the scratch, which the single-query kernel (no maxima of its own) must not read
    base = _exact_run(ctx, db, 10)[0]
    blank = X.ExactDb("blank", db.lineages, db.ref_win, db.ref_seqs, [X.no_kmer_query(30)] * len(db.queries))
    try:
        for G in (1, 2, 16):
            _exact_run(ctx, blank, 10)
            ctx.set_option(capi.RTX_OPT_HITCOUNT_GROUP, G)
            assert same_hits(base, _exact_run(ctx, db, 10)[0]), f"group {G}"
        ctx.set_option(capi.RTX_OPT_HITCOUNT_GROUP, 0)
        ctx.set_option(capi.RTX_OPT_SUB_BATCH, 2)
        assert same_hits(base, _exact_run(ctx, db, 10)[0]), "sub-batch 2"
    finally:
        ctx.set_option(capi.RTX_OPT_HITCOUNT_GROUP, 0)
        ctx.set_option(capi.RTX_OPT_SUB_BATCH, 0)


def test_best_hits_skip_mode_drops_exact_copies(ctx):
    """The skip read's exact copies (ids 3 and 600) are zeroed after the hit counting; the per-segment maxima still hold 80 for their
    segments, which therefore stay candidates and must be read -- and yield nothing at the copies."""
    db = _edge_db()
    for G in (0, 1):  # with the query-group kernel's stale maxima, and with no maxima at all
        ctx.set_option(capi.RTX_OPT_HITCOUNT_GROUP, G)
        try:
            for T in (1, 3, 10, 64):
                dev, ht, eo, eids = _exact_run(ctx, db, T, skip=True)
                assert sorted(eids[eo[1]: eo[2]]) == [3, 600]
                want = [db.counts(q) for q in db.queries]
                want[1][[3, 600]] = 0
                assert np.array_equal(dev.counts, np.array(want))
                assert_hits(dev, want, T, f"skip T={T}")
                n, ref, cnt = dev.best_hits
                assert ref[1, 0] == 1200 and cnt[1, 0] == 80
                assert 3 not in ref[1, : n[1]] and 600 not in ref[1, : n[1]]
            plain, *_ = _exact_run(ctx, db, 3)
            assert list(plain.best_hits[1][1, :3]) == [3, 600, 1200]
        finally:
            ctx.set_option(capi.RTX_OPT_HITCOUNT_GROUP, 0)


def test_best_hits_every_reference_tied(ctx):
    db = X.db_one_count()  # 77 references, all at 25
    for T in (10, 64):
        dev, *_ = _exact_run(ctx, db, T)
        n, ref, cnt = dev.best_hits
        assert n[0] == T and list(ref[0, :T]) == list(range(T)) and (cnt[0, :T] == 25).all()
    dev, *_ = _exact_run(ctx, db, 64)
    assert_hits(dev, dev.counts, 64)


# ---- 4. both strands ----------------------------------------------------------------------------------------------------------------
def test_best_hits_both_strands_equal_plus_mode_of_chosen_orientation(ctx, small):
    ds, ht, off, codes = small
    ctx.upload_tree(ht)
    flip = np.random.default_rng(99).random(len(off) - 1) < 0.5
    mixed = synth.reverse_complement_batch(off, codes, flip)
    for skip in (False, True):
        eo, eids = ht.exact_batch_both_strands(off, mixed)
        both = ctx.classify(off, mixed, eo, eids, skip_exact=skip, taps=("counts",), both_strands=True, best_hits=10)
        assert_hits(both, both.counts, 10, "both strands")
        oriented = synth.reverse_complement_batch(off, mixed, both.strand.astype(bool))
        plus = _classify(ctx, ht, off, oriented, skip, taps=("counts",), best_hits=10)
        assert same_hits(both, plus)
        assert both.strand[: ds.n_queries].astype(bool)[flip[: ds.n_queries]].mean() > 0.8


# ---- 5. refusals --------------------------------------------------------------------------------------------------------------------
def test_best_hits_refusals(ctx, small):
    ds, ht, off, codes = small
    ctx.upload_tree(ht)
    L = capi.device_lib()
    for bad in (-1, 65):
        assert L.rtx_ctx_set_option(ctx._h, capi.RTX_OPT_BEST_HITS, bad) == capi.RTX_ERR_INVALID
    nq = len(off) - 1
    n = np.zeros(nq, np.uint32)
    r = np.zeros(nq * 64, np.uint32)
    c = np.zeros(nq * 64, np.uint16)
    args = (n.ctypes.data_as(C.POINTER(C.c_uint32)), r.ctypes.data_as(C.POINTER(C.c_uint32)), c.ctypes.data_as(C.POINTER(C.c_uint16)))
    eo, eids = ht.exact_batch(off, codes)
    ctx.batch_upload(off, codes, eo, eids, best_hits=5)
    assert L.rtx_batch_best_hits(ctx._h, *args) == capi.RTX_ERR_INVALID  # uploaded, not downloaded
    assert L.rtx_shard_phase1(ctx._h) == capi.RTX_ERR_UNSUPPORTED
    assert L.rtx_shard_run(ctx._h) == capi.RTX_ERR_UNSUPPORTED
    assert b"reference-sharded" in L.rtx_last_error(ctx._h)
    ctx.batch_run()
    assert L.rtx_batch_best_hits(ctx._h, *args) == capi.RTX_ERR_INVALID  # run, not downloaded
    ctx.batch_download()
    assert L.rtx_batch_best_hits(ctx._h, *args) == capi.RTX_OK
    with pytest.raises(capi.RtxError) as ei:
        ctx.classify(off, codes, eo, eids, shard_root=0, best_hits=5)
    assert ei.value.code == capi.RTX_ERR_UNSUPPORTED
    plain = ctx.classify(off, codes, eo, eids)  # T = 0
    assert plain.best_hits is None
    assert L.rtx_batch_best_hits(ctx._h, *args) == capi.RTX_ERR_INVALID


# ---- 6. the host driver and the CLI on the committed diptera sample --------------------------------------------------------------------
GOLDEN_FASTA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "diptera_sample.fasta")


def _cli(*args):
    from raxtax_b200 import _build

    r = subprocess.run([_build.CLI_BIN, *map(str, args)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return r


def _hit_lines_from_taps(ctx, ht, labels, off, codes, T, both):
    eo, eids = (ht.exact_batch_both_strands if both else ht.exact_batch)(off, codes)
    dev = ctx.classify(off, codes, eo, eids, taps=("counts",), both_strands=both)
    lin = ht.lineages
    lines = []
    for q, (ids, c) in enumerate(expected_hits(dev.counts, T)):
        for k, (r, m) in enumerate(zip(ids, c)):
            l = f"{labels[q]}\t{k + 1}\t{lin[r]}\t{m}\t{dev.n_kmers[q]}\t{r}"
            lines.append(l + ("\t-" if dev.strand[q] else "\t+") if both else l)
    return lines


@pytest.mark.parametrize("tsv,both", [(False, False), (True, False), (False, True), (True, True)])
def test_cli_best_hits(ctx, tmp_path, tsv, both):
    q = capi.Queries.from_fasta(open(GOLDEN_FASTA).read())
    labels = q.labels
    off, codes = q.arrays()
    ht = capi.Tree.from_fasta(open(GOLDEN_FASTA).read())
    ctx.upload_tree(ht)
    flags = (["--tsv"] if tsv else []) + (["--strand", "both"] if both else [])
    _cli("-d", GOLDEN_FASTA, "-i", GOLDEN_FASTA, "-o", tmp_path / "plain", "--skip-db", *flags)
    _cli("-d", GOLDEN_FASTA, "-i", GOLDEN_FASTA, "-o", tmp_path / "hits", "--skip-db", "--best-hits", 5, *flags)
    for f in ["raxtax.out"] + (["raxtax.tsv"] if tsv else []):
        assert (tmp_path / "hits" / f).read_bytes() == (tmp_path / "plain" / f).read_bytes(), f
    assert not (tmp_path / "plain" / "raxtax.hits").exists()
    got = (tmp_path / "hits" / "raxtax.hits").read_text()
    want = _hit_lines_from_taps(ctx, ht, labels, off, codes, 5, both)
    assert got.endswith("\n") and got[:-1].split("\n") == want
    # the Python driver gives the same lines, right before each query's results, de-duplicated or not
    for env in ({}, {"RXH_NO_DEDUP": "1"}):
        old = {k: os.environ.get(k) for k in env}
        os.environ.update(env)
        try:
            sent, _, _, hits = capi.raxtax(ctx, q, ht, tsv=tsv, both_strands=both, best_hits=5)
        finally:
            for k, v in old.items():
                if v is None:
                    os.environ.pop(k, None)
        assert [h[0] for h in hits] == [s[0] for s in sent]
        assert sorted(l for _, h in hits if h for l in h.split("\n")) == sorted(want)
    # a run cut short mid-file resumes to the same raxtax.hits
    if not tsv:
        d = tmp_path / "cut"
        _cli("-d", GOLDEN_FASTA, "-i", GOLDEN_FASTA, "-o", d, "--skip-db", "--best-hits", 5, *flags)
        full_hits, full_out = (d / "raxtax.hits").read_bytes(), (d / "raxtax.out").read_bytes()
        done = (d / "raxtax.ckp").read_text().split("\n")[:150]
        (d / "raxtax.ckp").write_text("\n".join(done) + "\n")
        listed = {x.encode() for x in done}

        def cut(data):  # every line of the listed queries, a few of the next ones, then a torn line
            ls = data.split(b"\n")
            first = next(i for i, l in enumerate(ls) if l.split(b"\t", 1)[0] not in listed)
            return b"\n".join(ls[: first + 5]) + b"\n" + ls[first + 5][:7]

        (d / "raxtax.hits").write_bytes(cut(full_hits))
        (d / "raxtax.out").write_bytes(cut(full_out))
        _cli("-d", GOLDEN_FASTA, "-i", GOLDEN_FASTA, "-o", d, "--skip-db", "--best-hits", 5, *flags)
        assert (d / "raxtax.hits").read_bytes() == full_hits
        assert (d / "raxtax.out").read_bytes() == full_out
