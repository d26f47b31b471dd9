"""Deterministic synthetic barcode data for the BASELINE.json configs (SURVEY.md §8(d), Appendix D).

COI-like (650 bp, codon-position rate heterogeneity) and 16S-like (1500 bp, conserved backbone with nine
variable blocks) reference sets with 6-rank lineages `p:,c:,o:,f:,g:,s:` plus a query mix of exact copies,
near copies, unseen species and junk.  The substitution model is hierarchical (one round of per-site
substitutions per taxonomic rank) and calibrated so that the mean shared-8-mer fraction rho between a query
and a random reference lands in 0.15-0.30, as measured on the reference's example data (rho = 0.223).

Codes are raxtax's 4-bit one-hot codes (parser.rs:11-34): A=1 C=2 G=4 T=8, IUPAC = OR of members.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

BASE_CODES = np.array([1, 2, 4, 8], np.uint8)  # A C G T
COMPOSITION = np.array([0.263, 0.169, 0.143, 0.425])  # A C G T measured on example/diptera_queries.fasta
TWO_FOLD = np.array([3, 5, 6, 9, 10, 12], np.uint8)  # M R S W Y K
CODE_TO_CHAR = {1: "A", 2: "C", 4: "G", 8: "T", 9: "W", 6: "S", 3: "M", 12: "K", 5: "R", 10: "Y", 14: "B", 13: "D",
                11: "H", 7: "V", 15: "N"}

SEED_BASE = 0xB2000000

CONFIGS = {
    # name: (n_refs, n_queries, length, kind)
    "tiny": (600, 64, 300, "coi"),
    "small": (5000, 256, 650, "coi"),
    "c2": (100_000, 10_000, 650, "coi"),
    "c3": (1_000_000, 200_000, 650, "coi"),
    "c4": (500_000, 100_000, 1500, "16s"),
    "c5": (8_000_000, 1_000_000, 650, "coi"),
}
CONFIG_SEED = {"tiny": 10, "small": 11, "c2": 2, "c3": 3, "c4": 4, "c5": 5}


@dataclass
class Dataset:
    name: str
    ref_lineages: list  # N strings (unsorted, as they would appear in a FASTA)
    ref_off: np.ndarray  # u64[N+1]
    ref_codes: np.ndarray  # u8
    query_labels: list
    query_off: np.ndarray
    query_codes: np.ndarray
    meta: dict = field(default_factory=dict)

    @property
    def n_refs(self):
        return len(self.ref_lineages)

    @property
    def n_queries(self):
        return len(self.query_labels)

    def ref_seq(self, i):
        return self.ref_codes[int(self.ref_off[i]): int(self.ref_off[i + 1])]

    def query_seq(self, i):
        return self.query_codes[int(self.query_off[i]): int(self.query_off[i + 1])]

    def ref_fasta(self, width=60) -> str:
        return _fasta([f"R{i};tax={l};" for i, l in enumerate(self.ref_lineages)], self.ref_off, self.ref_codes, width)

    def query_fasta(self, width=60) -> str:
        return _fasta(self.query_labels, self.query_off, self.query_codes, width)


def _fasta(labels, off, codes, width):
    lut = np.full(256, ord("N"), np.uint8)
    for k, v in CODE_TO_CHAR.items():
        lut[k] = ord(v)
    chars = lut[codes]
    out = []
    for i, lab in enumerate(labels):
        s = chars[int(off[i]): int(off[i + 1])].tobytes().decode()
        out.append(">" + lab)
        for j in range(0, len(s), width):
            out.append(s[j: j + width])
    return "\n".join(out) + "\n"


def _site_rates(length, kind, rng):
    """Per-site relative substitution rates (mean about 1)."""
    pos = np.arange(length)
    if kind == "coi":
        codon = np.array([0.5, 0.2, 2.3])[pos % 3]
        # conserved / variable stretches: real COI keeps whole motifs fixed, which is what makes rho ~0.2
        region = np.empty(length)
        i = 0
        conserved = True
        while i < length:
            ln = int(rng.integers(8, 18)) if conserved else int(rng.integers(40, 100))
            region[i: i + ln] = 0.08 if conserved else 1.5
            conserved = not conserved
            i += ln
        return codon * region
    # 16S-like: conserved backbone (x0.3) with nine variable blocks of 60-100 bp (x3)
    rate = np.full(length, 0.3)
    starts = np.linspace(60, length - 160, 9).astype(int)
    for s in starts:
        ln = int(rng.integers(60, 101))
        rate[s: s + ln] = 3.0
    return rate


def _mutate(seqs, rate_per_site, rng):
    """One round of substitutions: each site redrawn from COMPOSITION with probability rate_per_site."""
    n, L = seqs.shape
    out = seqs.copy()
    chunk = max(1, (64 << 20) // max(L, 1))
    cum = np.cumsum(COMPOSITION)
    for a in range(0, n, chunk):
        b = min(n, a + chunk)
        mask = rng.random((b - a, L), dtype=np.float32) < rate_per_site[None, :].astype(np.float32)
        k = int(mask.sum())
        if k:
            draws = np.searchsorted(cum, rng.random(k)).clip(0, 3).astype(np.uint8)
            sub = out[a:b]
            sub[mask] = draws
    return out


def _assign_parents(n_child, n_parent, rng, skew=1.2):
    """Every parent gets >= 1 child; the rest follow a long-tailed preference."""
    n_parent = min(n_parent, n_child)
    w = 1.0 / np.arange(1, n_parent + 1) ** skew
    rng.shuffle(w)
    extra = rng.choice(n_parent, size=n_child - n_parent, p=w / w.sum())
    par = np.concatenate([np.arange(n_parent), extra])
    par.sort(kind="stable")
    return par


def generate_clades(name, n_clades, n_refs=None, n_queries=None, seed=None) -> Dataset:
    """A large reference set as `n_clades` diverged copies of one base set of n_refs / n_clades references: clade c carries the base
    lineages under its own phylum labels and the base sequences with 4 % of the bases substituted (so that no sequence is shared
    between clades and the 8-mer sharing across clades is that of distant relatives).  8 M references by the full hierarchical model
    take ~5 minutes and 20 GB of temporaries; this takes the base set's time plus a few seconds per clade.  Queries: the base set's
    query mix, each query assigned to a random clade and mutated like that clade's references where it copies one."""
    cfg = CONFIGS[name]
    n_refs = n_refs or cfg[0]
    n_queries = cfg[1] if n_queries is None else n_queries
    seed = SEED_BASE + CONFIG_SEED[name] if seed is None else seed
    base = generate(name, n_refs=n_refs // n_clades, n_queries=n_queries, length=cfg[2], kind=cfg[3], seed=seed, measure=False)
    rng = np.random.default_rng(seed + 7919)
    cum = np.cumsum(COMPOSITION)
    ref_parts, lin, lens = [], [], (base.ref_off[1:] - base.ref_off[:-1]).astype(np.int64)
    # substitution pattern per clade: a fixed set of alignment columns re-drawn (a clade-specific "ancestral" change), applied to
    # every sequence of the clade alike, references and the queries derived from them -- exact copies stay exact copies
    col_sub = [None] * n_clades
    pos_in_seq = (np.arange(len(base.ref_codes), dtype=np.int64) - np.repeat(base.ref_off[:-1].astype(np.int64), lens))
    for c in range(n_clades):
        codes = base.ref_codes.copy()
        if c:
            cols = rng.random(cfg[2]) < 0.04
            new_base = BASE_CODES[np.searchsorted(cum, rng.random(cfg[2])).clip(0, 3)]
            col_sub[c] = (cols, new_base)
            hit = cols[pos_in_seq] & (codes < 15) & np.isin(codes, BASE_CODES)
            codes[hit] = new_base[pos_in_seq[hit]]
        ref_parts.append(codes)
        lin += [l if c == 0 else l.replace("p:P", f"p:X{c}P", 1) for l in base.ref_lineages]
    ref_codes = np.concatenate(ref_parts)
    ref_off = np.zeros(len(lin) + 1, np.uint64)
    ref_off[1:] = np.cumsum(np.tile(lens, n_clades))
    # queries
    q_codes = base.query_codes.copy()
    q_lens = (base.query_off[1:] - base.query_off[:-1]).astype(np.int64)
    q_clade = rng.integers(0, n_clades, base.n_queries)
    q_pos = (np.arange(len(q_codes), dtype=np.int64) - np.repeat(base.query_off[:-1].astype(np.int64), q_lens))
    q_of = np.repeat(q_clade, q_lens)
    for c in range(1, n_clades):
        cols, new_base = col_sub[c]
        hit = (q_of == c) & cols[np.minimum(q_pos, cfg[2] - 1)] & np.isin(q_codes, BASE_CODES)
        q_codes[hit] = new_base[q_pos[hit]]
    meta = dict(base.meta, n_refs=len(lin), n_clades=n_clades, note="clade copies of a base set (synth.generate_clades)")
    return Dataset(name, lin, ref_off, ref_codes, base.query_labels, base.query_off, q_codes, meta=meta)


def generate(name="c2", n_refs=None, n_queries=None, length=None, kind=None, seed=None, measure=True) -> Dataset:
    if name == "c5" and n_refs is None and length is None and kind is None:
        return generate_clades("c5", 8, n_queries=n_queries, seed=seed)
    cfg = CONFIGS.get(name)
    if cfg is not None:
        n_refs = n_refs or cfg[0]
        n_queries = cfg[1] if n_queries is None else n_queries
        length = length or cfg[2]
        kind = kind or cfg[3]
        seed = SEED_BASE + CONFIG_SEED[name] if seed is None else seed
    assert n_refs and length and kind and seed is not None
    rng = np.random.default_rng(seed)
    site = _site_rates(length, kind, rng)

    # ---- taxonomy sizes (Appendix D: families : genera : species : seqs = 1 : 12.5 : 44 : 75)
    n_fam = max(1, round(n_refs / 75))
    n_gen = max(n_fam, round(n_refs * 12.5 / 75))
    n_spe = max(n_gen, round(n_refs * 44 / 75))
    n_spe = min(n_spe, n_refs)
    n_ord = min(40, n_fam)
    n_cla = min(6, n_ord)
    n_phy = min(2, n_cla)
    sizes = [n_phy, n_cla, n_ord, n_fam, n_gen, n_spe]
    # branch rates per rank (phylum, class, order, family, genus, species) then individual
    rates = [0.02, 0.02, 0.02, 0.013, 0.018, 0.053]
    rate_ind = 0.018
    if kind == "16s":
        rates = [r * 0.8 for r in rates]
        rate_ind *= 0.8

    cum = np.cumsum(COMPOSITION)
    root = np.searchsorted(cum, rng.random(length)).clip(0, 3).astype(np.uint8)[None, :]
    parents = []  # parents[l][i] = parent index at level l-1 of node i at level l
    seqs = root
    for lvl, n in enumerate(sizes):
        n_par = 1 if lvl == 0 else sizes[lvl - 1]
        par = _assign_parents(n, n_par, rng) if lvl else np.zeros(n, np.int64)
        parents.append(par)
        seqs = _mutate(seqs[par], np.clip(rates[lvl] * site, 0, 0.75), rng)
    species_seqs = seqs
    genus_of_species = parents[5]
    ref_species = _assign_parents(n_refs, n_spe, rng)
    ref2 = _mutate(species_seqs[ref_species], np.clip(rate_ind * site, 0, 0.75), rng)  # values 0..3

    # lineage strings
    chain = [np.arange(n_spe)]
    for lvl in range(5, 0, -1):
        chain.append(parents[lvl][chain[-1]])
    chain = chain[::-1]  # [phylum.., species] index per species
    prefixes = ["p:P", "c:C", "o:O", "f:F", "g:G", "s:S"]
    species_lineage = [",".join(prefixes[l] + str(int(chain[l][s])) for l in range(6)) for s in range(n_spe)]

    # ---- duplicates: ~0.5 % of refs copy another ref's sequence (same species mostly, a few across genera)
    n_dup = int(round(n_refs * 0.005))
    dup_pairs = []
    if n_dup:
        src = rng.integers(0, n_refs, n_dup)
        for s in src:
            if rng.random() < 0.9:
                same = np.nonzero(ref_species == ref_species[s])[0] if n_refs <= 20000 else None
                if same is not None and len(same) > 1:
                    d = int(rng.choice(same))
                else:  # neighbouring ref in the sorted-by-species order is usually the same species
                    d = int(min(n_refs - 1, s + 1))
            else:
                d = int(rng.integers(0, n_refs))
            if d != s:
                ref2[d] = ref2[s]
                dup_pairs.append((int(s), d))

    # ---- reference lengths: 20 % of refs lose up to 8 trailing bases
    ref_len = np.full(n_refs, length, np.int64)
    short = rng.random(n_refs) < 0.2
    ref_len[short] -= rng.integers(1, 9, int(short.sum()))
    ref_codes2d = BASE_CODES[ref2]
    # ambiguity codes: 0.1 % N, 0.02 % two-fold
    amb = rng.random(ref_codes2d.shape, dtype=np.float32)
    ref_codes2d[amb < 0.001] = 15
    m2 = (amb >= 0.001) & (amb < 0.0012)
    ref_codes2d[m2] = TWO_FOLD[rng.integers(0, 6, int(m2.sum()))]
    # duplicates must stay byte-identical including ambiguity codes and length
    for s, d in dup_pairs:
        ref_codes2d[d] = ref_codes2d[s]
        ref_len[d] = ref_len[s]

    # shuffle reference order so that the host-side lineage sort is actually exercised
    perm = rng.permutation(n_refs)
    ref_species_p = ref_species[perm]
    ref_len_p = ref_len[perm]
    ref_codes2d = ref_codes2d[perm]
    ref_off = np.zeros(n_refs + 1, np.uint64)
    ref_off[1:] = np.cumsum(ref_len_p)
    keep = np.arange(length)[None, :] < ref_len_p[:, None]
    ref_codes = np.ascontiguousarray(ref_codes2d[keep])
    ref_lineages = [species_lineage[s] for s in ref_species_p]

    # ---- queries
    nq = n_queries
    kinds = rng.choice(4, size=nq, p=[0.20, 0.50, 0.25, 0.05])
    q_rows = np.zeros((nq, length), np.uint8)
    q_len = np.full(nq, length, np.int64)
    src_ref = rng.integers(0, n_refs, nq)
    # exact copies
    e = kinds == 0
    q_rows[e] = ref_codes2d[src_ref[e]]
    q_len[e] = ref_len_p[src_ref[e]]
    # near copies: 1 % substitutions on the 2-bit sequence of a reference (ambiguity codes of the ref kept)
    n_ = kinds == 1
    if n_.any():
        base = ref_codes2d[src_ref[n_]].copy()
        mask = rng.random(base.shape, dtype=np.float32) < 0.01
        base[mask] = BASE_CODES[np.searchsorted(cum, rng.random(int(mask.sum()))).clip(0, 3)]
        q_rows[n_] = base
        q_len[n_] = ref_len_p[src_ref[n_]]
    # unseen species under an existing genus
    u = kinds == 2
    if u.any():
        genus_seqs_idx = genus_of_species[ref_species_p[src_ref[u]]]
        # recompute genus-level sequences lazily: mutate the species sequence again with species+individual rate
        base = species_seqs[ref_species_p[src_ref[u]]]
        base = _mutate(base, np.clip((rates[5] * 2 + rate_ind) * site, 0, 0.75), rng)
        q_rows[u] = BASE_CODES[base]
        del genus_seqs_idx
    # junk: unrelated random sequence, or a reference with runs of N
    j = np.nonzero(kinds == 3)[0]
    for qi in j:
        if rng.random() < 0.5:
            q_rows[qi] = BASE_CODES[np.searchsorted(cum, rng.random(length)).clip(0, 3)]
        else:
            row = ref_codes2d[src_ref[qi]].copy()
            for _ in range(int(rng.integers(1, 4))):
                a = int(rng.integers(0, length - 20))
                row[a: a + int(rng.integers(5, 60))] = 15
            q_rows[qi] = row
            q_len[qi] = ref_len_p[src_ref[qi]]
        if rng.random() < 0.1:
            q_len[qi] = int(rng.integers(0, 12))  # very short reads incl. shorter than one 8-mer
    q_off = np.zeros(nq + 1, np.uint64)
    q_off[1:] = np.cumsum(q_len)
    keepq = np.arange(length)[None, :] < q_len[:, None]
    q_codes = np.ascontiguousarray(q_rows[keepq])
    q_labels = [f"Q{i}|kind{int(kinds[i])}" for i in range(nq)]

    ds = Dataset(name, ref_lineages, ref_off, ref_codes, q_labels, q_off, q_codes,
                 meta=dict(seed=int(seed), n_refs=int(n_refs), n_queries=int(nq), length=int(length), kind=kind,
                           taxa=dict(zip(["phyla", "classes", "orders", "families", "genera", "species"], map(int, sizes))),
                           n_dup_pairs=len(dup_pairs)))
    if measure:
        ds.meta.update(measure_rho(ds, rng))
    return ds


# complement of a 4-bit code: the bit-reversed nibble (A1 <-> T8, C2 <-> G4, R5 <-> Y10, N15 <-> N15, ...)
COMPLEMENT = np.array([int(f"{c:04b}"[::-1], 2) for c in range(16)], np.uint8)


def reverse_complement(codes: np.ndarray) -> np.ndarray:
    """Reverse complement of one sequence of 4-bit codes."""
    return COMPLEMENT[np.asarray(codes, np.uint8)[::-1] & 15]


def reverse_complement_batch(off: np.ndarray, codes: np.ndarray, which=None) -> np.ndarray:
    """Packed sequences (codes[off[i]:off[i+1]]) with sequence i reverse-complemented where which[i] (all of them when which is
    None); the offsets do not change."""
    off = np.asarray(off, np.int64)
    codes = np.asarray(codes, np.uint8)
    n = len(off) - 1
    lens = off[1:] - off[:-1]
    sel = np.ones(n, bool) if which is None else np.asarray(which, bool)
    seg = np.repeat(np.arange(n), lens)
    pos = np.arange(len(codes), dtype=np.int64)
    flip = sel[seg]
    src = np.where(flip, off[:-1][seg] + off[1:][seg] - 1 - pos, pos)
    out = codes[src]
    return np.where(flip, COMPLEMENT[out & 15], out).astype(np.uint8)


def kmers_of(codes: np.ndarray) -> np.ndarray:
    """Sorted unique 8-mers of one sequence of 4-bit codes (utils.rs:27-40), numpy restatement used for data statistics."""
    if len(codes) < 8:
        return np.zeros(0, np.uint16)
    two = np.full(16, -1, np.int32)
    two[[1, 2, 4, 8]] = [0, 1, 2, 3]
    t = two[codes & 15]
    t = np.where(codes > 15, -1, t)
    n = len(codes) - 7
    val = np.zeros(n, np.int32)
    bad = np.zeros(n, bool)
    for jj in range(8):
        w = t[jj: jj + n]
        bad |= w < 0
        val |= np.where(w < 0, 0, w) << (14 - 2 * jj)
    return np.unique(val[~bad]).astype(np.uint16)


def measure_rho(ds: Dataset, rng=None, n_q=24, n_r=1500) -> dict:
    """Mean shared-8-mer fraction between sampled queries and sampled references, and distinct-count statistics."""
    rng = rng or np.random.default_rng(1)
    qs = rng.choice(ds.n_queries, size=min(n_q, ds.n_queries), replace=False) if ds.n_queries else []
    rs = rng.choice(ds.n_refs, size=min(n_r, ds.n_refs), replace=False)
    ref_sets = [kmers_of(ds.ref_seq(r)) for r in rs]
    fr, dd, ks = [], [], []
    for q in qs:
        kq = kmers_of(ds.query_seq(q))
        if len(kq) == 0:
            continue
        present = np.zeros(65536, bool)
        present[kq] = True
        cnt = np.array([int(present[s].sum()) for s in ref_sets])
        fr.append(cnt.mean() / len(kq))
        dd.append(len(np.unique(cnt)))
        ks.append(len(kq))
    return dict(rho=float(np.mean(fr)) if fr else 0.0, distinct_counts_sampled=float(np.mean(dd)) if dd else 0.0,
                mean_K=float(np.mean(ks)) if ks else 0.0)
