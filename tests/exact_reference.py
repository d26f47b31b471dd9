"""Exact references for hit counting and the probability tables, on databases cut from one de Bruijn sequence.

The linear de Bruijn sequence B(4, 8) has 65 543 bases and each of its 65 536 8-mer windows occurs once.  A query that is the
substring with windows [a, b) and a reference that is the substring with windows [s, e) therefore share exactly
|[a, b) ∩ [s, e)| 8-mers: the hit counts, the histograms and K of every query are known in closed form, and any histogram
{m: h[m]} can be laid out as a database.

`exact_probs` states prob.rs:8-103 in mpmath at 50 significant digits (no underflow, no truncation): the normalised P(m) of
every count a query's histogram holds and the global signal of lineage.rs:86-90.  It is a helper module, not a test file:
tests/test_exact_reference_cpu.py checks it, and the oracle, against known values; tests/test_gpu_exact_reference.py holds
the CUDA kernels to it.
"""
from __future__ import annotations

import functools
import math
from dataclasses import dataclass, field

import mpmath  # a missing package must fail loudly: torch's sympy dependency brings it
import numpy as np
from mpmath.libmp import from_int, mpf_add, mpf_div, mpf_mul, mpf_mul_int, mpf_pow_int, round_nearest

from raxtax_b200 import synth

DIGITS = 50
N_WINDOWS = 4 ** 8
N_BASES = N_WINDOWS + 7
E_CUT = 70.0        # the device drops E(i) < e^-70 (kernels.cuh kEcut)
TAIL_NATS = 40.0    # and a row's tail once ln pmf < -(40 + ln h) (kTailNats)
UNDERFLOW = -745.0  # forward rows start at the first pmf above e^-745


# ---- the sequence ------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=1)
def de_bruijn() -> np.ndarray:
    """The linear de Bruijn sequence B(4, 8) as 4-bit codes (synth.BASE_CODES): 65 543 bases, every 8-mer once."""
    k, n = 4, 8
    a = [0] * (k * n)
    seq = []

    def db(t, p):  # Fredricksen-Kessler-Maiorana: concatenated Lyndon words in lexicographic order
        if t > n:
            if n % p == 0:
                seq.extend(a[1: p + 1])
        else:
            a[t] = a[t - p]
            db(t + 1, p)
            for j in range(a[t - p] + 1, k):
                a[t] = j
                db(t + 1, t)

    db(1, 1)
    cyc = np.array(seq, np.int64)
    assert len(cyc) == N_WINDOWS
    return synth.BASE_CODES[np.concatenate([cyc, cyc[: n - 1]])]


def window_seq(s: int, e: int) -> np.ndarray:
    """The substring whose 8-mer windows are [s, e)."""
    assert 0 <= s < e <= N_WINDOWS
    return de_bruijn()[s: e + 7]


# ---- databases -----------------------------------------------------------------------------------------------------------------
@dataclass
class Query:
    codes: np.ndarray
    win: tuple | None  # (a, b): windows [a, b); None: no 8-mer at all (K = 0)
    name: str = ""

    @property
    def K(self) -> int:
        return 0 if self.win is None else self.win[1] - self.win[0]


@dataclass
class ExactDb:
    """References in sorted order (device reference id == construction order) and the queries laid out on them."""
    name: str
    lineages: list
    ref_win: np.ndarray  # [N, 2] windows [s, e) of each reference; s == e: no 8-mer (a sequence shorter than 8 bases)
    ref_seqs: list
    queries: list = field(default_factory=list)

    @property
    def n_refs(self) -> int:
        return len(self.lineages)

    def packed_refs(self):
        off = np.zeros(self.n_refs + 1, np.uint64)
        off[1:] = np.cumsum([len(s) for s in self.ref_seqs])
        return off, np.concatenate(self.ref_seqs).astype(np.uint8)

    def packed_queries(self):
        return pack([q.codes for q in self.queries])

    def counts(self, q: Query) -> np.ndarray:
        """Closed form: the hit count of every reference is the overlap of its window interval with the query's."""
        if q.win is None:
            return np.zeros(self.n_refs, np.uint16)
        a, b = q.win
        ov = np.minimum(self.ref_win[:, 1], b) - np.maximum(self.ref_win[:, 0], a)
        return np.clip(ov, 0, None).astype(np.uint16)

    def hist(self, q: Query) -> np.ndarray:
        return np.bincount(self.counts(q).astype(np.int64), minlength=q.K + 1)[: q.K + 1]


def pack(seqs):
    """list of code arrays -> (offsets u64[n + 1], codes u8[total])"""
    off = np.zeros(len(seqs) + 1, np.uint64)
    off[1:] = np.cumsum([len(s) for s in seqs])
    return off, (np.concatenate(seqs).astype(np.uint8) if len(seqs) else np.zeros(0, np.uint8))


def hist_dict(h) -> dict:
    return {int(m): int(v) for m, v in enumerate(h) if v}


class Layout:
    """Lays out references with prescribed hit counts against prescribed query intervals.  Every reference is a substring of
    the de Bruijn sequence; its count against any query of the database follows from the window intervals alone."""

    def __init__(self, seed):
        self.rng = np.random.default_rng(seed)
        self.refs = []  # (s, e, codes)

    def overlap(self, a, b, c, slack=4):
        """A reference sharing exactly c windows with [a, b) (0 < c < b - a; c == b - a gives a superstring, never the same
        sequence): a random stretch of c windows of the query, extended outside the query where it touches an end."""
        K = b - a
        assert 0 < c <= K
        if c == K:
            s, e = a - 1 - int(self.rng.integers(0, slack)), b + int(self.rng.integers(0, slack))
        else:
            s0 = a + int(self.rng.integers(0, K - c + 1))
            s, e = s0, s0 + c
            if s == a:
                s -= int(self.rng.integers(0, slack))
            if e == b:
                e += int(self.rng.integers(0, slack))
        s, e = max(s, 0), min(e, N_WINDOWS)
        self.refs.append((s, e, window_seq(s, e)))

    def exact(self, a, b):
        self.refs.append((a, b, window_seq(a, b)))

    def outside(self, lo, hi, n):
        """n references whose windows lie in [lo, hi): count 0 against every query outside that range; every ninth one is a
        sequence shorter than 8 bases instead."""
        for _ in range(n):
            if self.rng.random() < 1 / 9:
                ln = int(self.rng.integers(1, 8))
                s = int(self.rng.integers(lo, hi))
                self.refs.append((s, s, de_bruijn()[s: s + ln].copy()))
                continue
            ln = int(self.rng.integers(1, 24))
            s = int(self.rng.integers(lo, hi - ln))
            self.refs.append((s, s + ln, window_seq(s, s + ln)))

    def finish(self, name, queries, main=None, stride=8) -> ExactDb:
        """Orders the references so that the ones with the highest count against `main` (a query index; default 0) sit on both
        sides of the 8-reference block and 512-reference segment boundaries (positions = 0, 7, 8, 511 mod 512 of every
        `stride`-th segment), the other high ones packed in front, the rest shuffled behind; then groups them into lineage
        nodes of 1-5, 13, 37, 700 and 1 100 references."""
        N = len(self.refs)
        win = np.array([(s, e) for s, e, _ in self.refs], np.int64).reshape(N, 2)
        q = queries[0 if main is None else main]
        a, b = q.win
        cnt = np.clip(np.minimum(win[:, 1], b) - np.maximum(win[:, 0], a), 0, None)
        by_count = np.lexsort((self.rng.random(N), -cnt))  # descending count, ties in random order
        special = sorted(p for s in range(0, (N + 511) // 512, stride) for p in (512 * s, 512 * s + 7, 512 * s + 8, 512 * s + 511) if p < N)
        n_high = int((cnt > 0).sum())
        n_spec = min(len(special), n_high)
        pos = np.full(N, -1, np.int64)
        pos[by_count[:n_spec]] = special[:n_spec]
        free = np.setdiff1d(np.arange(N), special[:n_spec])
        rest = by_count[n_spec:]
        hi_rest, lo_rest = rest[: n_high - n_spec], rest[n_high - n_spec:]
        lo_rest = lo_rest[self.rng.permutation(len(lo_rest))]
        pos[np.concatenate([hi_rest, lo_rest]).astype(np.int64)] = free
        order = np.argsort(pos)
        sizes = [1, 2, 3, 4, 5, 13, 1, 5, 37, 2, 700, 4, 3, 1100]
        lineages, node, i, k = [], 0, 0, 0
        while i < N:
            n = sizes[k % len(sizes)]
            for j in range(i, min(N, i + n)):
                lineages.append(f"root,g{node // 7:05d},n{node:06d},r{j:07d}")
            i += n
            node += 1
            k += 1
        return ExactDb(name, lineages, win[order], [self.refs[o][2] for o in order], list(queries))


def window_query(a, b, name="") -> Query:
    return Query(window_seq(a, b).copy(), (a, b), name)


def no_kmer_query(length, name="") -> Query:
    """K = 0: all-N (length >= 8) or shorter than 8 bases."""
    codes = np.full(length, 15, np.uint8) if length >= 8 else de_bruijn()[100: 100 + length].copy()
    return Query(codes, None, name)


# ---- the catalogue ---------------------------------------------------------------------------------------------------------------
def _lay(L: Layout, a, b, hist: dict, zero_lo, zero_hi):
    for m, h in sorted(hist.items()):
        if m == 0:
            L.outside(zero_lo, zero_hi, h)
        else:
            for _ in range(h):
                L.overlap(a, b, m)


def db_kat(with_full=True) -> ExactDb:
    """prob.rs:229: K = 400 and one reference per count 0..400 (without the count-400 one: the slow branch with D = 400); the
    same database serves reads with K = 0 (all-N, and 5 bases), 1, 2 and 3."""
    a, b = 1000, 1400
    L = Layout(1 if with_full else 2)
    _lay(L, a, b, {m: 1 for m in range(0, 401 if with_full else 400)}, 30000, 31000)
    qs = [window_query(a, b, "kat"), no_kmer_query(20, "all-N"), no_kmer_query(5, "5 bases"), window_query(a + 17, a + 18, "K=1"),
          window_query(b - 2, b, "K=2"), window_query(a + 150, a + 153, "K=3")]
    return L.finish("kat" if with_full else "kat-slow", qs)


def db_peak() -> ExactDb:
    """A read-like peak: h[0] = 50 000, a few references at 20 / 100 / 300 and one at 420 (K = 600); 50 k references are 25
    reference tiles.  Sub-reads of the peak read and reads off every reference fill a batch of 19."""
    a, b = 5000, 5600
    L = Layout(3)
    _lay(L, a, b, {0: 50000, 20: 3, 100: 4, 300: 2, 420: 1}, 20000, 60000)
    qs = [window_query(a, b, "peak")]
    rng = np.random.default_rng(31)
    for j in range(13):
        x = int(rng.integers(a - 30, b - 40))
        qs.append(window_query(x, x + int(rng.integers(20, min(560, b + 30 - x))), f"sub {j}"))
    qs += [window_query(10000 + 90 * j, 10000 + 90 * j + 40 + 37 * j, f"no hit {j}") for j in range(3)]
    qs += [no_kmer_query(40, "all-N"), window_query(a + 5, a + 6, "K=1")]
    return L.finish("peak", qs)


def db_heavy() -> ExactDb:
    """A heavy low block: K = 800, h[10] = 200 000, h[40] = 20 000, h[60] = h[61] = 300, h[62] = 1 (220 601 references, more than
    one CSR tile).  The mass cut puts m_min near 60 and whole 512-reference segments are dropped by their maxima."""
    a, b = 3000, 3800
    L = Layout(5)
    _lay(L, a, b, {10: 200000, 40: 20000, 60: 300, 61: 300, 62: 1}, 0, 1)
    qs = [window_query(a, b, "heavy"), window_query(a + 100, a + 700, "heavy sub 1"), window_query(a + 400, b, "heavy sub 2"),
          window_query(a, a + 90, "heavy sub 3")]
    return L.finish("heavy", qs, stride=16)


def db_ties() -> ExactDb:
    """Exact ties: a read whose references share two counts only (0 and 37, K = 60), and reads that see one count only."""
    a, b = 2000, 2060
    L = Layout(7)
    _lay(L, a, b, {0: 120, 37: 50}, 40000, 41000)
    qs = [window_query(a, b, "two counts"), window_query(40000 - 50, 40000 - 10, "all at 0"),
          window_query(a + 23, a + 60, "sub"), window_query(a + 23, a + 24, "K=1 sub")]
    return L.finish("ties", qs)


def db_one_count() -> ExactDb:
    """Every reference at one count m = 25 < K = 60: uniform probabilities."""
    a, b = 7000, 7060
    L = Layout(8)
    for _ in range(77):
        L.overlap(a, b, 25)
    return L.finish("one-count", [window_query(a, b, "one count")])


def db_dense() -> ExactDb:
    """A dense middle: K = 2 000, h[m] in [20, 80] for every even m in 900..1 100 and h[0] = 50 000; E wakes up late, and many rows
    are evaluated from the top."""
    a, b = 40000, 42000
    rng = np.random.default_rng(9)
    L = Layout(9)
    _lay(L, a, b, {0: 50000, **{m: int(rng.integers(20, 81)) for m in range(900, 1101, 2)}}, 0, 30000)
    return L.finish("dense", [window_query(a, b, "dense")])


def db_spread() -> ExactDb:
    """A flat spread: K = 2 001, one reference at each of 168 counts 0, 12, 24, .., 2 000 (more distinct counts than threads)."""
    a, b = 12000, 14001
    L = Layout(10)
    _lay(L, a, b, {m: 1 for m in range(0, 2001, 12)}, 30000, 40000)
    return L.finish("spread", [window_query(a, b, "spread")])


def db_long() -> ExactDb:
    """Large K: 6 500 with D = 50 and 12 000 with D = 4 (three counts and 0)."""
    a1, b1, a2, b2 = 100, 6600, 20000, 32000
    rng = np.random.default_rng(11)
    L = Layout(11)
    ms = sorted(set(int(x) for x in rng.integers(2500, 6499, 60)))[:47]
    _lay(L, a1, b1, {**{m: int(rng.integers(1, 4)) for m in ms}, 6498: 1, 6450: 2}, 50000, 60000)
    _lay(L, a2, b2, {5000: 2, 9000: 1, 11990: 1}, 50000, 60000)
    L.outside(50000, 60000, 20)
    return L.finish("long", [window_query(a1, b1, "K=6500"), window_query(a2, b2, "K=12000")])


def db_huge() -> ExactDb:
    """K = 47 500 with five counts and 0 (D = 6)."""
    a, b = 9000, 56500
    L = Layout(12)
    _lay(L, a, b, {0: 30, 30000: 2, 41000: 1, 47000: 2, 47400: 1, 47499: 1}, 0, 8000)
    return L.finish("huge", [window_query(a, b, "K=47500")])


# reads of at most 1 426 bases: the probability tables of their batch fit the first shared-memory layout
LAYOUT_A_DBS = ("kat", "kat-slow", "peak", "heavy", "ties", "one-count")
CATALOGUE = {"kat": lambda: db_kat(True), "kat-slow": lambda: db_kat(False), "peak": db_peak, "heavy": db_heavy, "ties": db_ties,
             "one-count": db_one_count, "dense": db_dense, "spread": db_spread, "long": db_long, "huge": db_huge}


@functools.lru_cache(maxsize=None)
def catalogue_db(name) -> ExactDb:
    db = CATALOGUE[name]()
    assert all(s <= e for s, e in db.ref_win)
    return db


# ---- prob.rs:8-103 in exact arithmetic ---------------------------------------------------------------------------------------------
def pmf_mode(K, t, m):
    """The device's closed form of the mode of pmf_m (kernels.cuh pmf_mode)."""
    if K <= 2:
        return t
    num = m * t - K + m - t + 1
    if num < 0:
        return 0
    return min(t, num // (K - 2) + 1)


@dataclass
class ExactProbs:
    K: int
    P: dict           # m -> normalised P(m), mpmath mpf
    signal: object    # global signal (mpf)
    fast: bool        # some reference has count K: prob.rs:24-26
    i0: int | None    # slow branch: first i with ln E(i) > -70
    rows: dict        # slow branch, m >= 1: m -> (mode, tail end, ln pmf(0), class)

    def P_float(self, m) -> float:
        return float(self.P[m])


def _mpf(x):
    return mpmath.mpf(x)


def _first_true(lo, hi, pred):
    """smallest i in [lo, hi) with pred(i), else hi; pred is monotone (false.. true..)"""
    while lo < hi:
        mid = (lo + hi) // 2
        if pred(mid):
            hi = mid
        else:
            lo = mid + 1
    return lo


@functools.lru_cache(maxsize=None)
def _exact_probs(K, hist_items, N):
    hist = dict(hist_items)
    rnd = round_nearest
    t = K // 2
    with mpmath.workdps(DIGITS):
        prec = mpmath.mp.prec
        one = from_int(1)
        fast = hist.get(K, 0) > 0
        rows = {}
        i0 = None
        if fast:  # only_last_pmf (prob.rs:105-119)
            Ct = mpmath.binomial(K + t - 1, t)
            raw = {m: (_mpf(1) if m == K else _mpf(0) if m == 0 else mpmath.binomial(m + t - 1, t) / Ct) for m in hist}
        else:
            T = mpmath.binomial(K + t - 1, t)

            def row(m):
                """pmf_m(0..t) by the exact ratio recurrence, and the running cmf"""
                p = mpmath.binomial(K - m + t - 1, t) / T
                p = p._mpf_
                pm, cm, c = [], [], None
                for i in range(t + 1):
                    c = p if c is None else mpf_add(c, p, prec, rnd)
                    pm.append(p)
                    cm.append(c)
                    if i < t:
                        p = mpf_div(mpf_mul_int(p, (m + i) * (t - i), prec, rnd), from_int((i + 1) * (K - m + t - i - 1)), prec, rnd)
                return pm, cm

            E = [one] * (t + 1)
            cache = {}
            for m, h in hist.items():
                if m == 0:  # pmf = delta(i, 0): cmf == 1
                    continue
                pm, cm = row(m)
                cache[m] = (pm, cm)
                for i in range(t + 1):
                    E[i] = mpf_mul(E[i], mpf_pow_int(cm[i], h, prec, rnd), prec, rnd)
            raw = {}
            for m in hist:
                if m == 0:
                    raw[m] = mpmath.mpf(E[0])
                    continue
                pm, cm = cache[m]
                s = from_int(0)
                for i in range(t + 1):
                    s = mpf_add(s, mpf_mul(pm[i], mpf_div(E[i], cm[i], prec, rnd), prec, rnd), prec, rnd)
                raw[m] = mpmath.mpf(s)
            # coverage diagnostics from exact arithmetic
            ln = lambda x: mpmath.log(mpmath.mpf(x))
            i0 = _first_true(0, t + 1, lambda i: ln(E[i]) > -E_CUT)  # E is non-decreasing
            for m, h in hist.items():
                if m == 0:
                    continue
                pm, _ = cache[m]
                mode = pmf_mode(K, t, m)
                thr = -(TAIL_NATS + math.log(h))
                hi = _first_true(mode + 1, t + 1, lambda i: ln(pm[i]) < thr)  # the pmf falls above its mode
                lp0 = float(mpmath.log(mpmath.mpf(pm[0])))
                if i0 > mode:
                    cls = "finished" if hi <= i0 else "top"
                else:
                    cls = "forward-underflow" if lp0 < UNDERFLOW else "forward"
                rows[m] = (mode, hi, lp0, cls)
        S = mpmath.fsum(hist[m] * raw[m] for m in hist)
        P = {m: raw[m] / S for m in hist}
        inv = mpmath.mpf(1) / N
        signal = mpmath.sqrt(mpmath.fsum(hist[m] * (P[m] - inv) ** 2 for m in hist))
    return ExactProbs(K, P, signal, fast, i0, rows)


def exact_probs(K, hist) -> ExactProbs:
    """prob.rs:8-103 at DIGITS significant digits for one query: K unique 8-mers, t = K // 2 trials, hist = {count: references} or a
    count-indexed array.  Cached per histogram."""
    h = hist if isinstance(hist, dict) else hist_dict(hist)
    h = {int(m): int(v) for m, v in h.items() if v}
    assert all(0 <= m <= K for m in h)
    return _exact_probs(int(K), tuple(sorted(h.items())), sum(h.values()))


def bar(K) -> float:
    """The relative part r(K) of the bar |P_dev - P_exact| <= r(K) P_exact + 1e-15: the device's ln pmf is a difference of ln n!
    values as large as lnGamma(K + t + 1), so its absolute error grows with it (measured at 1.7e-12 for K = 600, 2.3e-11 for
    K = 6 000, 1.2e-10 for K = 65 535); r(K) leaves a 30-80x margin."""
    return 1e-14 * math.lgamma(K + K // 2 + 1)


BAR_ABS = 1e-15


def bar_ratio(K, got, exact) -> float:
    """|got - exact| / (r(K) exact + 1e-15): <= 1 passes the bar."""
    e = float(exact)
    return abs(float(got) - e) / (bar(K) * abs(e) + BAR_ABS)

