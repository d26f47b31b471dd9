"""The CUDA path against exact arithmetic on de Bruijn databases (tests/exact_reference.py).

Hit counts, histograms and K are known in closed form and must come back bit-exact.  The normalised P(m) of every count a query's
histogram holds, and the global signal, must lie within

    |P_dev - P_exact| <= r(K) P_exact + 1e-15,   r(K) = 1e-14 lnGamma(K + floor(K/2) + 1)

of the mpmath statement of prob.rs (exact_reference.bar: the device builds ln pmf from differences of ln n! values as large as
lnGamma(K + t + 1)).  The result lines (raw confidences: the one-exact-match override is covered by the parity tests) must be the
oracle's lineage evaluation of the exact probabilities, up to the tie and rounding-boundary outcomes tests/parity.py tolerates.

The catalogue runs through every memory layout of the probability kernel -- the longest read of a batch picks it: per-warp sums
with ln n! in shared memory (reads up to 1 426 bases), one shared sum array updated with atomics (up to 6 402), tables in global
scratch (longer) -- through the hit-count launch space (queries per CTA, reference tile groups, the CSR variant, partial query
groups, the single-query kernel with its histogram in global memory), at every bit-plane boundary, in skip mode and with both
strands."""
import numpy as np
import pytest

from raxtax_b200 import capi, synth
from tests import exact_reference as X
from tests import parity
from tests.test_gpu_parity import _same_outputs

pytestmark = pytest.mark.gpu
TAPS = ("counts", "hist", "kmers", "probs")
WORST = {}  # layout -> (worst |dP| / bar, where)


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


_trees = {}


def _trees_of(oracle, db):
    if db.name not in _trees:
        _trees.clear()  # one database's trees at a time: the large ones hold hundreds of MB
        off, codes = db.packed_refs()
        ot = oracle.Tree.new(db.lineages, db.ref_seqs)
        _trees[db.name] = (capi.Tree.new(db.lineages, off, codes), ot, parity.TolerantChecker(ot.flatten(), ot.num_tips))
    return _trees[db.name]


def _upload(oracle, ctx, db):
    ht, ot, chk = _trees_of(oracle, db)
    ctx.upload_tree(ht)
    assert ctx.n_refs == db.n_refs
    return ht, ot, chk


def _classify(ctx, ht, qs, skip=False, **kw):
    off, codes = X.pack([q.codes for q in qs])
    eo, eids = ht.exact_batch(off, codes)
    return ctx.classify(off, codes, eo, eids, skip_exact=skip, raw_conf=True, taps=TAPS, **kw)


def _companion(length):
    return X.Query(np.full(length, 15, np.uint8), None, f"all-N {length}")


def _check(db, ot, chk, qs, dev, layout, zeroed=None):
    """Counts, histograms and K bit-exact; P(m) and the global signal within the bar; result lines = the oracle's evaluation of
    the exact probabilities.  zeroed[i]: references whose count query i's skip mode zeroes.  Returns the number of queries whose
    lines needed tie / rounding tolerance."""
    tolerated = 0
    for i, q in enumerate(qs):
        c = db.counts(q)
        if zeroed is not None:
            c[zeroed[i]] = 0
        h = np.bincount(c.astype(np.int64), minlength=q.K + 1)
        assert int(dev.n_kmers[i]) == q.K, q.name
        assert np.array_equal(dev.counts[i], c), f"{db.name} / {q.name}: hit counts"
        assert np.array_equal(dev.hist[i, : q.K + 1], h), f"{db.name} / {q.name}: histogram"
        ep = X.exact_probs(q.K, h)
        for m in ep.P:
            r = X.bar_ratio(q.K, dev.probs[i, m], ep.P[m])
            assert r <= 1.0, f"{db.name} / {q.name} ({layout}): P({m}) = {dev.probs[i, m]!r}, exact {ep.P_float(m)!r}"
            if r > WORST.get(layout, (-1.0,))[0]:
                WORST[layout] = (r, f"{db.name} / {q.name}, K = {q.K}, m = {m}")
        assert X.bar_ratio(q.K, dev.global_signal[i], ep.signal) <= 1.0, f"{db.name} / {q.name} ({layout}): global signal"
        pr = np.zeros(q.K + 1)
        for m in ep.P:
            pr[m] = ep.P_float(m)
        p_ref = pr[c]
        exp = ot.evaluate(p_ref).for_query(0)
        got = dev.for_query(i)
        if not parity.results_equal(exp, got):
            assert chk.acceptable(p_ref, got, exp), f"{db.name} / {q.name} ({layout}): result lines {got} vs {exp}"
            tolerated += 1
    return tolerated


def _report(layout, tolerated, nq):
    r, where = WORST.get(layout, (0.0, "-"))
    print(f"{layout}: {nq} queries, {tolerated} tolerated; worst |dP| / bar so far {r:.3g} ({where})")


# ---- the catalogue through the three layouts of the probability kernel ----------------------------------------------------------
LAYOUTS = [("A", 0, None), ("B", 3000, None), ("C group", 9000, "hitcount_group_kernel<16> (2 queries per CTA)"),
           ("C single, global histogram", 48000, "hitcount_bitrows_kernel<16>")]


@pytest.mark.parametrize("name", X.LAYOUT_A_DBS)
def test_catalogue_in_every_layout(oracle, ctx, name):
    """The reads of at most 1 426 bases alone, then with an all-N companion read (K = 0: no other query's histogram changes) of
    3 000, 9 000 and 48 000 bases, which moves the batch to the shared-atomics layout, to global scratch with two queries per
    hit-count CTA, and to global scratch with the single-query hit-count kernel and its histogram in global memory."""
    db = X.catalogue_db(name)
    assert max(len(q.codes) for q in db.queries) <= 1426
    ht, ot, chk = _upload(oracle, ctx, db)
    for layout, comp, kernel in LAYOUTS:
        qs = list(db.queries) + ([_companion(comp)] if comp else [])
        dev = _classify(ctx, ht, qs)
        if kernel is not None:
            assert ctx.hitcount_kernel_name() == kernel
        _report(layout, _check(db, ot, chk, qs, dev, layout), len(qs))


@pytest.mark.parametrize("name,layout", [("dense", "B"), ("spread", "B"), ("long", "C group"), ("huge", "C single, global histogram")])
def test_catalogue_long_reads(oracle, ctx, name, layout):
    """K = 2 000 and 2 001 (shared-atomics layout by themselves), 6 500 and 12 000, and 47 500 (global scratch)."""
    db = X.catalogue_db(name)
    ht, ot, chk = _upload(oracle, ctx, db)
    dev = _classify(ctx, ht, db.queries)
    _report(layout, _check(db, ot, chk, db.queries, dev, layout), len(db.queries))


# ---- hit counting: the launch space ---------------------------------------------------------------------------------------------
def _differences(a, b):
    """What differs bit for bit between two runs: result lines and signals, and the taps.  The probability tap is compared where
    the histogram is non-zero, the part it defines (a query's table row keeps what an earlier query of its sub-batch slot left
    beyond its own counts)."""
    held = a.hist > 0
    same = {"result lines": _same_outputs(a, b), "K": np.array_equal(a.n_kmers, b.n_kmers), "counts": np.array_equal(a.counts, b.counts),
            "hist": np.array_equal(a.hist, b.hist), "kmers": np.array_equal(a.kmers, b.kmers),
            "probs": np.array_equal(a.probs[held], b.probs[held])}
    return [k for k, v in same.items() if not v]


def test_hitcount_launch_space(oracle, ctx):
    """19 reads on 50 010 references (25 reference tiles): every queries-per-CTA choice (partial last query groups included), one,
    three and the default number of tiles per CTA (25, 9 and one reference tile group), the CSR variant and sub-batches of 7 give
    outputs bit-identical to the default run, which itself is exact."""
    db = X.catalogue_db("peak")
    qs = db.queries
    assert len(qs) == 19 and db.n_refs >= 20000
    ht, ot, chk = _upload(oracle, ctx, db)
    ref = _classify(ctx, ht, qs)
    assert ctx.hitcount_kernel_name() == "hitcount_group_kernel<10> (4 queries per CTA)"
    _check(db, ot, chk, qs, ref, "A")
    runs = 0
    try:
        for G in (0, 1, 2, 3, 5, 8, 13, 16):
            for tiles in (0, 1, 3):
                ctx.set_option(capi.RTX_OPT_HITCOUNT_GROUP, G)
                ctx.set_option(capi.RTX_OPT_HITCOUNT_MAX_TILES, tiles)
                dev = _classify(ctx, ht, qs)
                want = "hitcount_bitrows_kernel<10>" if G == 1 else f"hitcount_group_kernel<10> ({G or 4} queries per CTA)"
                assert ctx.hitcount_kernel_name() == want, (G, tiles)
                assert not _differences(ref, dev), (G, tiles, _differences(ref, dev))
                runs += 1
        ctx.set_option(capi.RTX_OPT_HITCOUNT_GROUP, 0)
        ctx.set_option(capi.RTX_OPT_HITCOUNT_MAX_TILES, 0)
        ctx.set_option(capi.RTX_OPT_SUB_BATCH, 7)  # 7 + 7 + 5 queries: partial groups of 3 and 1
        dev = _classify(ctx, ht, qs)
        assert ctx.hitcount_kernel_name() == "hitcount_group_kernel<10> (4 queries per CTA)"
        assert not _differences(ref, dev), ("sub-batches of 7", _differences(ref, dev))
        ctx.set_option(capi.RTX_OPT_SUB_BATCH, 0)
        ctx.set_option(capi.RTX_OPT_KEEP_CSR, 1)
        ctx.set_option(capi.RTX_OPT_HITCOUNT_VARIANT, capi.RTX_HITCOUNT_CSR)
        off, codes = db.packed_refs()
        ctx.upload_tree(capi.Tree.new(db.lineages, off, codes, eager_kmer_map=True))
        dev = _classify(ctx, ht, qs)
        assert ctx.hitcount_kernel_name() == "hitcount_csr_kernel"
        assert not _differences(ref, dev), ("CSR", _differences(ref, dev))
    finally:
        for opt, v in ((capi.RTX_OPT_HITCOUNT_GROUP, 0), (capi.RTX_OPT_HITCOUNT_MAX_TILES, 0), (capi.RTX_OPT_SUB_BATCH, 0),
                       (capi.RTX_OPT_HITCOUNT_VARIANT, capi.RTX_HITCOUNT_BITROWS), (capi.RTX_OPT_KEEP_CSR, 0)):
            ctx.set_option(opt, v)
    print(f"{runs + 2} launch configurations bit-identical to the default")


# ---- bit-plane boundaries -----------------------------------------------------------------------------------------------------
NP_BOUNDS = {256: 10, 1024: 11, 2048: 13, 8192: 16}
NP_BELOW = {256: 8, 1024: 10, 2048: 11, 8192: 13}


@pytest.fixture(scope="module")
def np_db():
    """For every kmax in NP_BOUNDS a read with exactly kmax 8-mers (kmax + 7 bases) and its superstring among the references, so
    that a count equals kmax; the same read one base shorter; and three shorter sub-reads."""
    L = X.Layout(21)
    qs, starts = [], {}
    a = 100
    for kmax in NP_BOUNDS:
        starts[kmax] = a
        L.overlap(a, a + kmax, kmax)
        for c in (kmax - 1, kmax // 2, 3):
            L.overlap(a, a + kmax, c)
        qs += [X.window_query(a, a + kmax, f"K={kmax}"), X.window_query(a, a + kmax - 1, f"K={kmax - 1}"),
               X.window_query(a + 2, a + 40, "sub 1"), X.window_query(a + 7, a + kmax // 3, "sub 2"), X.window_query(a + 1, a + 9, "sub 3")]
        a += kmax + 50
    L.outside(a + 100, a + 2000, 300)
    return L.finish("np", qs)


@pytest.mark.parametrize("kmax", list(NP_BOUNDS))
def test_bit_plane_boundaries(oracle, ctx, np_db, kmax):
    db = np_db
    ht, ot, chk = _upload(oracle, ctx, db)
    j = list(NP_BOUNDS).index(kmax) * 5
    for top, NP in ((j, NP_BOUNDS[kmax]), (j + 1, NP_BELOW[kmax])):
        qs = [db.queries[top]] + db.queries[j + 2: j + 5]
        assert max(len(q.codes) for q in qs) - 7 == qs[0].K and qs[0].K in (kmax, kmax - 1)
        dev = _classify(ctx, ht, qs)
        assert ctx.hitcount_kernel_name().startswith(f"hitcount_group_kernel<{NP}>")
        assert int(dev.counts[0].max()) == qs[0].K  # the superstring: a count of exactly K
        _check(db, ot, chk, qs, dev, f"NP {NP}")


# ---- skip mode ---------------------------------------------------------------------------------------------------------------
def test_skip_mode_fast_branch_through_superstring(oracle, ctx):
    """--skip-exact-matches zeroes the exact copy of a read.  With a superstring among the references a count of K survives and
    the fast branch stays; without one the read falls to the slow branch."""
    L = X.Layout(31)
    (a1, b1), (a2, b2) = (500, 800), (2000, 2300)
    L.exact(a1, b1)
    L.exact(a1, b1)
    L.overlap(a1, b1, b1 - a1)
    L.exact(a2, b2)
    for c in (299, 250, 120, 7, 1):
        L.overlap(a1, b1, c)
        L.overlap(a2, b2, c)
    L.outside(5000, 6000, 40)
    qs = [X.window_query(a1, b1, "exact + superstring"), X.window_query(a2, b2, "exact only"), X.window_query(a1 + 5, a1 + 100, "sub"),
          X.window_query(a2 + 1, b2, "sub of exact only")]
    db = L.finish("skip", qs)
    ht, ot, chk = _upload(oracle, ctx, db)
    dev = _classify(ctx, ht, qs, skip=True)
    zeroed = [np.array([np.array_equal(s, q.codes) for s in db.ref_seqs]) for q in qs]
    assert zeroed[0].sum() == 2 and zeroed[1].sum() == 1 and not zeroed[2].any()
    _check(db, ot, chk, qs, dev, "A", zeroed)
    assert dev.hist[0, 300] == 1 and dev.probs[0, 300] > 0.0  # fast branch through the superstring
    assert dev.hist[1, 300] == 0
    c1 = db.counts(qs[1])
    c1[zeroed[1]] = 0
    assert not X.exact_probs(300, np.bincount(c1.astype(np.int64), minlength=301)).fast


# ---- both strands ------------------------------------------------------------------------------------------------------------
def test_both_strands_pick_the_original(oracle, ctx):
    """The reads of the KAT database reverse-complemented, classified with both strands: the device picks the orientation by
    M(rc(s)) > M(s) (closed-form counts of the original, the oracle's of the reverse complement), and every read it turns gives
    the taps and result lines of the plain run of the original, bit for bit."""
    db = X.catalogue_db("kat")
    qs = db.queries
    ht, ot, chk = _upload(oracle, ctx, db)
    plain = _classify(ctx, ht, qs)
    off, codes = db.packed_queries()
    rc = synth.reverse_complement_batch(off, codes)
    o = ot.classify(off, rc, threads=4, chunk_size=4, want_counts=True)
    m_orig = np.array([db.counts(q).max() for q in qs])
    rule = (m_orig > o["counts"].max(axis=1)).astype(np.uint8)
    eo, eids = ht.exact_batch_both_strands(off, rc)
    dev = ctx.classify(off, rc, eo, eids, raw_conf=True, taps=TAPS, both_strands=True)
    assert np.array_equal(dev.strand, rule)
    assert rule.sum() >= 4 and rule[1] == 0 and rule[2] == 0  # the K = 0 reads tie and stay as given
    for i in np.nonzero(rule)[0]:
        assert np.array_equal(dev.counts[i], plain.counts[i]) and np.array_equal(dev.hist[i], plain.hist[i])
        assert np.array_equal(dev.probs[i], plain.probs[i]) and dev.global_signal[i] == plain.global_signal[i]
        a, b = dev.for_query(i), plain.for_query(i)
        assert len(a) == len(b) and all(x[0] == y[0] and np.array_equal(x[1], y[1]) and x[2] == y[2] for x, y in zip(a, b)), i
