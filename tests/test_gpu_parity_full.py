"""Parity at the benchmarked sizes (run on the B200 box): BASELINE config 1 in full (the reference's example file as its own
database, both modes), the exact batch bench.py times on config 2, and configs 3 / 4 at their full reference counts -- all against the
CPU oracle over the same inputs, counts bit-exact, result lines identical up to the two documented ambiguities (tests/parity.py)."""
import gzip
import os

import numpy as np
import pytest

from raxtax_b200 import capi, synth
from tests import parity

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


def _example_text():
    """The reference repository's example/diptera_queries.fasta, stored whole (tests/golden/make_diptera_full.py)."""
    return gzip.open(os.path.join(GOLDEN, "diptera_queries.fasta.gz"), "rt").read()


@pytest.mark.parametrize("skip", [False, True])
def test_config1_whole_example_file_as_its_own_database(oracle, ctx, skip):
    """All 7 868 records of example/diptera_queries.fasta against themselves (SURVEY.md 8(c)): default mode exercises the exact-match
    log / override / multi-match paths on real data, --skip-exact-matches the slow probability branch."""
    text = _example_text()
    ot = oracle.Tree.from_fasta(text)
    ht = capi.Tree.from_fasta(text)
    labels, q_off, q_codes = oracle.parse_queries(text)
    nq = len(labels)
    assert nq == 7868 and ot.num_tips == 7868 == ht.num_tips
    ctx.upload_tree(ht)
    eo, eids = ht.exact_batch(q_off, q_codes)
    dev = ctx.classify(q_off, q_codes, eo, eids, skip_exact=skip, taps=("counts", "hist", "kmers", "probs"))
    o = ot.classify(q_off, q_codes, skip_exact=skip, threads=os.cpu_count() or 4, chunk_size=50, want_counts=True, want_probs=True, want_kmers=True)
    assert np.array_equal(o["K"], dev.n_kmers)
    assert np.array_equal(o["counts"], dev.counts), "hit counts"
    for q in range(0, nq, 97):
        K = int(o["K"][q])
        assert np.array_equal(o["kmers"][q, :K], dev.kmers[q, :K])
        assert np.array_equal(parity.hist_from_counts(o["counts"][q], K), dev.hist[q, : K + 1])
    assert np.array_equal(o["nexact"], eo[1:] - eo[:-1]), "exact-match sets"
    worst = 0.0
    for q in range(0, nq, 13):
        worst = max(worst, float(np.max(np.abs(dev.probs[q][dev.counts[q].astype(np.int64)] - o["probs"][q]))))
    assert worst <= 1e-9, f"probabilities differ from the oracle by {worst:.3e}"
    checker = parity.TolerantChecker(ot.flatten(), ot.num_tips)
    ok, tol, bad = parity.compare_batch(o, dev, nq, checker, o["probs"])
    assert not bad, f"{len(bad)} queries differ beyond tie / rounding tolerance, first {bad[:5]}"
    assert tol <= nq // 20
    print(f"config 1 ({'skip' if skip else 'default'}): {ok} of {nq} queries identical to the oracle, {tol} within tie / rounding tolerance, max |dP| {worst:.1e}")
    # the text the drop-in driver sends, against the oracle's formatting of its own results
    qs = capi.Queries.from_fasta(text)
    sent, logs, _ = capi.raxtax(ctx, qs, ht, skip_exact_matches=skip)
    assert [s[0] for s in sent] == labels
    exp = parity.lines_by_query(oracle.format_results(ot, o["results"], labels), labels)
    parity.assert_text_parity([s[1].split("\n") for s in sent], exp, o, ot, what=f"config 1 text ({'skip' if skip else 'default'})")
    assert sum(1 for lvl, _ in logs if lvl == 3) == (0 if skip else int(o["nexact"].sum()))


def test_config2_the_benchmarked_batch_against_the_oracle(oracle, ctx):
    """The first 512 queries of the exact 10 000-query batch `bench.py --workload c2` times, against the oracle over the same 100 000
    references: counts bit-exact, result lines identical."""
    ds = synth.generate("c2", measure=False)  # what bench.load_workload("c2", 10000) generates
    assert ds.n_queries == 10_000 and ds.n_refs == 100_000
    n = 512
    ht = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes)
    ctx.upload_tree(ht)
    eo, eids = ht.exact_batch(ds.query_off, ds.query_codes)
    dev_all = ctx.classify(ds.query_off, ds.query_codes, eo, eids)  # the whole batch, as the bench runs it
    q_off = ds.query_off[: n + 1]
    q_codes = ds.query_codes[: int(q_off[-1])]
    dev = ctx.classify(q_off, q_codes, eo[: n + 1], eids[: int(eo[n])], taps=("counts", "probs"))
    n_lines = int(dev.result_begin[-1])
    assert np.array_equal(dev_all.result_begin[: n + 1], dev.result_begin) and np.array_equal(dev_all.first_ref[:n_lines], dev.first_ref)
    assert np.array_equal(dev_all.confidence[:n_lines], dev.confidence) and np.array_equal(dev_all.local_signal[:n_lines], dev.local_signal)
    ot = parity.oracle_tree_from_ds(oracle, ds)
    o = ot.classify(q_off, q_codes, threads=os.cpu_count() or 4, chunk_size=8, want_counts=True, want_probs=True)
    assert np.array_equal(o["K"], dev.n_kmers) and np.array_equal(o["counts"], dev.counts), "hit counts of the benchmarked batch"
    checker = parity.TolerantChecker(ot.flatten(), ot.num_tips)
    ok, tol, bad = parity.compare_batch(o, dev, n, checker, o["probs"])
    assert not bad, f"{len(bad)} queries of the benchmarked batch differ from the oracle, first {bad[:3]}"
    assert tol <= n // 20
    print(f"c2 bench batch: {ok} of {n} queries identical to the oracle, {tol} within tie / rounding tolerance")
    # ... and through the driver, in text
    qs = capi.Queries.new(ds.query_labels[:n], q_off, q_codes)
    sent, _, _ = capi.raxtax(ctx, qs, ht, chunk_size=200)
    exp = parity.lines_by_query(oracle.format_results(ot, o["results"], ds.query_labels[:n]), ds.query_labels[:n])
    parity.assert_text_parity([s[1].split("\n") for s in sent], exp, o, ot, what="c2 bench batch text")
