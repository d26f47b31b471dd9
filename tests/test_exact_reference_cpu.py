"""The exact references of tests/exact_reference.py, checked without a GPU: the de Bruijn databases give the hit counts the closed
form says (through the oracle and the host library), the mpmath statement of prob.rs reproduces the known values, and the oracle
agrees with it on every catalogue histogram within the bar the device is held to."""
import numpy as np
import pytest

from raxtax_b200 import capi
from tests import exact_reference as X


def test_de_bruijn_windows_are_distinct():
    d = X.de_bruijn()
    assert len(d) == X.N_BASES and set(np.unique(d)) == set(int(c) for c in (1, 2, 4, 8))
    two = np.zeros(16, np.int64)
    two[[1, 2, 4, 8]] = [0, 1, 2, 3]
    v = two[d]
    val = np.zeros(X.N_WINDOWS, np.int64)
    for j in range(8):
        val = val * 4 + v[j: j + X.N_WINDOWS]
    assert len(np.unique(val)) == X.N_WINDOWS


@pytest.mark.parametrize("name", list(X.CATALOGUE))
def test_builder_counts_match_oracle(oracle, name):
    db = X.catalogue_db(name)
    ot = oracle.Tree.new(db.lineages, db.ref_seqs)
    assert ot.lineages == db.lineages  # already in sorted order: reference ids are construction order
    off, codes = db.packed_refs()
    assert capi.Tree.new(db.lineages, off, codes).lineages == db.lineages
    q_off, q_codes = db.packed_queries()
    o = ot.classify(q_off, q_codes, threads=4, chunk_size=4, want_counts=True)
    for i, q in enumerate(db.queries):
        assert int(o["K"][i]) == q.K, q.name
        assert np.array_equal(o["counts"][i], db.counts(q)), q.name
    main = db.queries[0]
    if name == "kat":
        assert X.hist_dict(db.hist(main)) == {m: 1 for m in range(401)}
    if name == "kat-slow":
        assert X.hist_dict(db.hist(main)) == {m: 1 for m in range(400)}
    if name == "heavy":
        assert X.hist_dict(db.hist(main)) == {10: 200000, 40: 20000, 60: 300, 61: 300, 62: 1} and db.n_refs > 65536


def test_reference_reproduces_known_values():
    """prob.rs:229-235 and SURVEY App. B: K = 400, t = 200, one reference per count 0..400."""
    ep = X.exact_probs(400, {m: 1 for m in range(401)})
    assert ep.fast
    assert abs(sum(ep.P.values()) - 1) < 1e-40
    got = [ep.P_float(m) for m in (398, 399, 400)]
    assert got == pytest.approx([0.148515837432, 0.223146911519, 0.335], abs=1e-12)
    assert all(ep.P[m] <= ep.P[m + 1] for m in range(400))
    # K = 0: every count equals K, uniform; K = 1 without a hit: the m == 0 row alone, uniform
    for K, h in ((0, {0: 5}), (1, {0: 4}), (20, {0: 3})):
        ep = X.exact_probs(K, h)
        assert ep.P_float(0) == pytest.approx(1 / sum(h.values()), rel=1e-15) and float(ep.signal) < 1e-40


def _all_histograms():
    for name in X.CATALOGUE:
        db = X.catalogue_db(name)
        for q in db.queries:
            yield name, db, q, db.hist(q)


def test_oracle_agrees_with_reference_within_bar(oracle):
    worst = (0.0, None)
    for name, db, q, h in _all_histograms():
        ep = X.exact_probs(q.K, h)
        c = db.counts(q)
        p = oracle.highest_hit_prob_per_reference(q.K, q.K // 2, c)
        first = {int(m): int(np.argmax(c == m)) for m in ep.P}
        for m, r in first.items():
            ratio = X.bar_ratio(q.K, p[r], ep.P[m])
            assert ratio <= 1.0, f"{name} / {q.name}: P({m}) = {p[r]!r}, exact {ep.P_float(m)!r}"
            worst = max(worst, (ratio, f"{name} / {q.name}, m = {m}"), key=lambda x: x[0])
        sig = np.sqrt(np.sum((p - 1.0 / db.n_refs) ** 2))
        assert X.bar_ratio(q.K, sig, ep.signal) <= 1.0, f"{name} / {q.name}: global signal"
    print(f"oracle vs exact: worst |dP| / bar = {worst[0]:.3g} ({worst[1]})")


def test_catalogue_coverage():
    classes, Ks, fast, D = set(), set(), False, []
    for _, _, q, h in _all_histograms():
        ep = X.exact_probs(q.K, h)
        classes |= {r[3] for r in ep.rows.values()}
        Ks.add(q.K)
        fast |= ep.fast
        D.append((len(ep.P), q.K))
    assert classes == {"finished", "top", "forward", "forward-underflow"}
    assert fast
    assert {0, 1, 2, 3} <= Ks and any(k % 2 for k in Ks if k > 3) and any(k % 2 == 0 for k in Ks if k > 3)
    assert any(d > 256 for d, _ in D) and any(d == k + 1 for d, k in D if k > 3)
