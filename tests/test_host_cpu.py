"""CPU-side tests (no GPU): the C++ host library against the reference's KATs and against the oracle, and the
C-ABI surface of both shared libraries (load + every symbol the headers declare; no compute calls)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from raxtax_b200 import _build, capi, synth
from tests.test_oracle_kats import KMER_KAT_CODES, REF_FASTA_KMERS, REF_FASTA_STR_PARSER

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module", autouse=True)
def _built():
    _build.build_all()


def _header_functions(path):
    text = open(path).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b((?:rtx|rxh)_[a-z0-9_]+)\s*\(", text)) - {"rxh_sender", "rxh_logger"})


def test_device_abi_exports_every_declared_symbol():
    names = _header_functions(os.path.join(ROOT, "include", "raxtax_b200.h"))
    assert sorted(names) == sorted(capi.DEVICE_SYMBOLS)
    lib = C.CDLL(_build.DEVICE_LIB)
    for n in names:
        assert hasattr(lib, n), n
    lib.rtx_abi_version.restype = C.c_int
    assert lib.rtx_abi_version() == 4


def test_host_abi_exports_every_declared_symbol():
    names = _header_functions(os.path.join(ROOT, "include", "raxtax_host.h"))
    assert sorted(names) == sorted(capi.HOST_SYMBOLS)
    lib = capi.host_lib()
    for n in names:
        assert hasattr(lib, n), n


def test_no_cpu_fallback_without_gpu():
    """Without a CUDA device the product must fail loudly instead of computing on the CPU."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(capi.RtxError) as ei:
        capi.Context(0)
    assert ei.value.code == capi.RTX_ERR_NO_DEVICE
    assert "no CPU fallback" in ei.value.msg


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "raxtax_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h", ".hpp")):
                src = open(os.path.join(dirpath, f), errors="replace").read()
                assert "oracle" not in src.lower(), f"{f} mentions the oracle"


# ---- reference KATs through the host library --------------------------------------------------------------------
def test_host_str_parser_kat():  # parser.rs:166-217
    tree = capi.Tree.from_fasta(REF_FASTA_STR_PARSER)
    assert list(tree.k_mer_map(0b1_0101_1111_1110)) == [0]
    assert list(tree.k_mer_map(0b11_0001_1001_1111)) == [1, 4, 5]
    assert list(tree.k_mer_map(0b110_0111_0011_1010)) == [3]
    assert tree.num_tips == 6
    assert tree.lineages[0].endswith("s:Species1") and tree.lineages[5].startswith("p:Phylum2")


def test_host_kmers_kat():  # parser.rs:235-299
    tree = capi.Tree.from_fasta(REF_FASTA_KMERS)
    assert list(tree.k_mer_map(0b1_0101_0110)) == [0, 4]
    assert list(tree.k_mer_map(0b101_0101_1010)) == [1, 4]
    assert list(tree.k_mer_map(0b1111_1100_0000_0001)) == [2, 3]


def test_host_query_parser_kat():  # parser.rs:219-233
    q = capi.Queries.from_fasta(">label1\nACGTWSMKRYBDHVN")
    off, codes = q.arrays()
    assert q.labels == ["label1"]
    assert list(codes) == [1, 2, 4, 8, 9, 6, 3, 12, 5, 10, 14, 13, 11, 7, 15]


def test_host_parser_errors():
    for text, msg in [("", "File is empty"), ("ACGT\n>x;tax=a,b;\nACGT", "Not a valid FASTA"), (">x;tax=a,b;\nACGU", "Unexpected character"),
                      (">x;taxon=a,b\nACGT", "taxonomical annotation"), (">x;tax=a,b;\n>y;tax=a,c;\nACGT", "does not match")]:
        with pytest.raises(capi.HostError, match=msg):
            capi.Tree.from_fasta(text)
    with pytest.raises(capi.HostError, match="File is empty"):
        capi.Queries.from_fasta("")


def _node_set_oracle(flat):
    """(lo, hi, type, depth) of the oracle's nodes minus childless Sequence leaves, children order preserved per parent."""
    keep = [i for i in range(len(flat["lo"])) if not (flat["type"][i] == 2 and flat["nchildren"][i] == 0)]
    return keep


def _compare_tree(orc_tree, host_tree):
    assert orc_tree.num_tips == host_tree.num_tips
    assert orc_tree.lineages == host_tree.lineages
    off_o, ids_o = orc_tree.csr()
    off_h, ids_h = host_tree.csr()
    assert np.array_equal(off_o, off_h)
    assert np.array_equal(ids_o, ids_h)
    # node structure: rebuild parent/child lists from the BFS arrays and compare with the oracle's pre-order tree
    ia = host_tree.index_arrays()
    flat = orc_tree.flatten()
    keep = _node_set_oracle(flat)
    assert len(keep) == len(ia["node_lo"])
    # walk both trees simultaneously
    o_children = {i: [] for i in range(len(flat["lo"]))}
    for i in range(1, len(flat["lo"])):
        o_children[int(flat["parent"][i])].append(i)
    keepset = set(keep)
    stack = [(0, 0)]
    while stack:
        o, h = stack.pop()
        assert (int(flat["lo"][o]), int(flat["hi"][o]), int(flat["type"][o])) == (int(ia["node_lo"][h]), int(ia["node_hi"][h]), int(ia["node_type"][h]))
        oc = [c for c in o_children[o] if c in keepset]
        cf, cc = int(ia["child_first"][h]), int(ia["child_count"][h])
        assert len(oc) == cc
        for j, c in enumerate(oc):
            stack.append((c, cf + j))
    # ref_levels
    assert list(ia["ref_levels"]) == [l.count(",") + 1 for l in host_tree.lineages]


def test_host_tree_matches_oracle_on_kat_fastas(oracle):
    for text in (REF_FASTA_STR_PARSER, REF_FASTA_KMERS):
        _compare_tree(oracle.Tree.from_fasta(text), capi.Tree.from_fasta(text))


def test_host_tree_matches_oracle_variable_depth_and_degenerate(oracle):
    lineages = [
        "Animalia,Chordata,Mammalia,Primates,Hominidae,Homo,Homo_sapiens", "Animalia,Chordata,Mammalia,Primates,Hominidae,Pan",
        "Animalia,Chordata,Mammalia,Carnivora,Canidae,Canis", "Animalia,Chordata,Mammalia,Carnivora,Doggo",
        "Animalia,Chordata,Mammalia,Mouse", "Animalia,Chordata,Mammalia,Carnivora,Felidae,Felis",
        "Animalia,Chordata,Mammalia,Carnivora,Felidae,Felis",
        "A,X", "A,X,X", "A,X,X,Y", "A,B", "A,B,C", "A,B!,C", "A,B-x,C", "Z", "Z", "",
    ]
    rng = np.random.default_rng(0)
    seqs = [synth.BASE_CODES[rng.integers(0, 4, 40)] for _ in lineages]
    off, codes = oracle.pack_sequences(seqs)
    _compare_tree(oracle.Tree.new(lineages, seqs), capi.Tree.new(lineages, off, codes))


def test_host_tree_matches_oracle_on_synthetic(oracle):
    ds = synth.generate("tiny")
    seqs = [ds.ref_seq(i) for i in range(ds.n_refs)]
    ot = oracle.Tree.new(ds.ref_lineages, seqs)
    ht = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes)
    _compare_tree(ot, ht)
    # exact-match map
    for q in range(ds.n_queries):
        s = ds.query_seq(q)
        assert list(ot.exact(s)) == list(ht.exact(s))
    eo, eids = ht.exact_batch(ds.query_off, ds.query_codes)
    assert eo[-1] == len(eids) and eo[-1] > 0
    # FASTA round trip through both parsers
    ot2 = oracle.Tree.from_fasta(ds.ref_fasta())
    ht2 = capi.Tree.from_fasta(ds.ref_fasta())
    _compare_tree(ot2, ht2)
    assert ot2.lineages == ot.lineages
    lab_o, off_o, codes_o = oracle.parse_queries(ds.query_fasta())
    hq = capi.Queries.from_fasta(ds.query_fasta())
    off_h, codes_h = hq.arrays()
    assert lab_o == hq.labels and np.array_equal(off_o, off_h) and np.array_equal(codes_o, codes_h)


def test_synth_kmers_match_oracle(oracle):
    ds = synth.generate("tiny", measure=False)
    for q in list(range(10)) + [ds.n_queries - 1]:
        assert np.array_equal(synth.kmers_of(ds.query_seq(q)), oracle.sequence_to_kmers(ds.query_seq(q)))
    assert list(synth.kmers_of(np.array(KMER_KAT_CODES, np.uint8))) == list(oracle.sequence_to_kmers(KMER_KAT_CODES))


def test_cli_exit_codes_without_gpu(tmp_path):
    """main.rs exit codes: NOINPUT for unreadable input; without a GPU the binary stops with TEMPFAIL instead of computing on the CPU."""
    import subprocess

    import torch

    # a missing database cannot be fingerprinted: Args::get_output fails -> CANTCREAT (main.rs:25-30, io.rs:31-33)
    r = subprocess.run([_build.CLI_BIN, "-d", "/nonexistent.fasta", "-i", "/nonexistent.fasta", "-o", str(tmp_path / "o1")], capture_output=True, text=True)
    assert r.returncode == 73
    r = subprocess.run([_build.CLI_BIN, "--only-db", "-d", "x", "-o", str(tmp_path / "o0")], capture_output=True, text=True)
    assert r.returncode == 73
    # neither a binary database nor FASTA -> NOINPUT (main.rs:61-71)
    bad = tmp_path / "bad.fasta"
    bad.write_text("this is not fasta\n")
    r = subprocess.run([_build.CLI_BIN, "-d", str(bad), "-i", str(bad), "-o", str(tmp_path / "o3")], capture_output=True, text=True)
    assert r.returncode == 66 and "Failed to parse" in r.stderr and "Not a valid FASTA file" in r.stderr
    if not torch.cuda.is_available():
        fasta = os.path.join(ROOT, "tests", "golden", "diptera_sample.fasta")
        r = subprocess.run([_build.CLI_BIN, "-d", fasta, "-i", fasta, "-o", str(tmp_path / "o2")], capture_output=True, text=True)
        assert r.returncode == 75 and "no CPU fallback" in r.stderr


def test_kmer_map_is_lazy_and_identical_to_the_oracles():
    """Tree.k_mer_map (tree.rs:41) is materialised on first use; content = the oracle's (parser.rs:166-217 style check on synthetic data)."""
    from oracle import oracle as orc
    from raxtax_b200 import synth

    ds = synth.generate("tiny", measure=False)
    ht = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes)
    assert not ht.has_kmer_map
    off, ids = ht.csr()
    assert ht.has_kmer_map
    ot = orc.Tree.new(ds.ref_lineages, [ds.ref_seq(i) for i in range(ds.n_refs)])
    ooff, oids = ot.csr()
    assert np.array_equal(off, ooff) and np.array_equal(ids, oids)
    eager = capi.Tree.new(ds.ref_lineages, ds.ref_off, ds.ref_codes, eager_kmer_map=True)
    assert eager.has_kmer_map
    eoff, eids = eager.csr()
    assert np.array_equal(off, eoff) and np.array_equal(ids, eids)


def test_cli_only_db_writes_the_reference_database_and_checkpoint(tmp_path):
    """--only-db needs no GPU: <prefix>/<stem>.bin in the reference's bincode layout + raxtax.json (io.rs:47-78,269-286; main.rs:73-102);
    a .bin passed as -d is loaded instead of parsed (parser.rs:37-44)."""
    import json
    import subprocess

    from tests import bincode_model as bm

    fasta = os.path.join(ROOT, "tests", "golden", "diptera_sample.fasta")
    prefix = tmp_path / "db"
    r = subprocess.run([_build.CLI_BIN, "--only-db", "-d", fasta, "-o", str(prefix)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    db = prefix / "diptera_sample.bin"
    t = bm.deserialize(db.read_bytes())
    assert t["num_tips"] == 400 and len(t["lineages"]) == 400 and t["lineages"] == sorted(t["lineages"], key=str.encode)
    assert len(t["k_mer_map"]) == 65536 and t["root"][0] == "root" and t["root"][1:3] == [0, 400]
    ck = json.loads((prefix / "raxtax.json").read_text())
    assert set(ck) == {"checkpoint_file", "progress_file", "db_fingerprint", "raw_confidence", "skip_exact_matches", "tsv"}
    assert ck["db_fingerprint"]["path"] == str(db) and ck["db_fingerprint"]["size"] == db.stat().st_size
    assert ck["progress_file"] == str(prefix / "raxtax.ckp") and ck["tsv"] is False
    # again into the same folder: the checkpoint is valid, the database is read back from the .bin, nothing is rebuilt
    before = db.stat().st_mtime_ns
    r = subprocess.run([_build.CLI_BIN, "--only-db", "-d", fasta, "-o", str(prefix)], capture_output=True, text=True)
    assert r.returncode == 0 and "Restarting from checkpoint" in r.stderr and db.stat().st_mtime_ns == before
    # the .bin as the database of a fresh run
    other = tmp_path / "other"
    r = subprocess.run([_build.CLI_BIN, "--only-db", "-d", str(db), "-o", str(other)], capture_output=True, text=True)
    assert r.returncode == 0 and not list(other.glob("*.bin"))
    # same content as parsing the FASTA
    a = capi.Tree.from_bin(db.read_bytes())
    b = capi.Tree.from_fasta(open(fasta).read())
    assert a.lineages == b.lineages
    ao, ai = a.csr()
    bo, bi = b.csr()
    assert np.array_equal(ao, bo) and np.array_equal(ai, bi)


def test_fixed_point_formatting_matches_libc():
    """rxh_format_fixed (the fast path behind every confidence and signal of a result line, lineage.rs:17-30) prints what "%.Nf"
    prints: the exact binary value rounded to nearest, ties to even -- Rust's `{:.N}`."""
    rng = np.random.default_rng(7)
    vals = [0.0, 1.0, 0.125, 0.375, 0.005, 0.015, 0.025, 0.995, 0.999995, 0.0000049999, 1.41421356, 0.5, 0.25, 1e-9, 123456.789, -0.0, -1.5,
            float("inf"), float("nan"), 1e12, 0.004999999999999999, 0.105, 2.675, 0.000005, 0.000015, 999999999.999999]
    r = rng.random(20000)
    vals += list(r) + list(np.round(r, 2)) + list(np.round(r, 5) + 0.5e-5) + list(np.round(r, 2) + 0.005) + list(r * 1.5)
    for v in vals:
        for prec in (2, 5):
            assert capi.format_fixed(v, prec) == "%.*f" % (prec, v), (v, prec)


def _tree_arrays(t):
    d = capi.IndexDesc()
    capi.host_lib().rxh_tree_index_desc(t._h, C.byref(d))
    nn, n = d.n_nodes, d.n_refs
    g = lambda p, k: np.ctypeslib.as_array(p, (k,)).copy()
    off = g(d.ref_seq_offsets, n + 1)
    return (g(d.node_lo, nn), g(d.node_hi, nn), g(d.node_type, nn), g(d.child_first, nn), g(d.child_count, nn), g(d.ref_levels, n), off,
            g(d.ref_seq_codes, int(off[-1])) if off[-1] else np.zeros(0, np.uint8))


@pytest.mark.parametrize("block,piece", [(None, None), ("64", "1"), ("1000", "200"), ("100000", "3000")])
def test_streamed_fasta_files_equal_in_memory_parse(tmp_path, monkeypatch, block, piece):
    """rxh_tree_from_file / rxh_queries_from_file (plain and gz, read in blocks, blocks cut into pieces parsed in parallel) give what
    the one-string parsers give; tiny blocks and pieces force every record across a block / piece boundary."""
    import gzip

    ds = synth.generate("tiny", measure=False)
    ref_txt = ds.ref_fasta().replace("\n>", "\n\n; a comment line\n   \n>", 3)  # blank / comment lines are dropped (parser.rs:53-57)
    q_txt = ds.query_fasta()
    want_t = capi.Tree.from_fasta(ref_txt)
    want_q = capi.Queries.from_fasta(q_txt)
    if block:
        monkeypatch.setenv("RXH_FASTA_BLOCK", block)
        monkeypatch.setenv("RXH_FASTA_PIECE", piece)
    for gz in (False, True):
        rp, qp = tmp_path / ("r.fasta" + (".gz" if gz else "")), tmp_path / ("q.fasta" + (".gz" if gz else ""))
        (gzip.open if gz else open)(rp, "wt").write(ref_txt)
        (gzip.open if gz else open)(qp, "wt").write(q_txt)
        t, was_db = capi.Tree.from_file(str(rp))
        assert not was_db and t.lineages == want_t.lineages
        for a, b in zip(_tree_arrays(t), _tree_arrays(want_t)):
            assert np.array_equal(a, b)
        q = capi.Queries.from_file(str(qp))
        assert q.labels == want_q.labels
        for a, b in zip(q.arrays(), want_q.arrays()):
            assert np.array_equal(a, b)
    # a binary database is recognised by content and loaded as such
    binp = tmp_path / "db.bin"
    want_t.save_bin(str(binp))
    t, was_db = capi.Tree.from_file(str(binp))
    assert was_db and t.lineages == want_t.lineages


def test_streamed_fasta_errors_match_the_parsers(tmp_path):
    cases = [("", "File is empty"), ("ACGT\n>x;tax=a,b;\nACGT", "Not a valid FASTA"), (">x;tax=a,b;\nACGU", "Unexpected character"),
             (">x;taxon=a,b\nACGT", "taxonomical annotation"), (">x;tax=a,b;\n>y;tax=a,c;\nACGT", "does not match"), ("\n  \n;c\n", "Not a valid FASTA")]
    for i, (text, msg) in enumerate(cases):
        p = tmp_path / f"e{i}.fasta"
        p.write_text(text)
        with pytest.raises(capi.HostError, match=msg):
            capi.Tree.from_file(str(p))
    with pytest.raises(capi.HostError, match="cannot read file"):
        capi.Tree.from_file(str(tmp_path / "missing.fasta"))
    # queries: empty records are merged into the next one, the last record is kept even when empty (parser.rs:138-147)
    p = tmp_path / "q.fasta"
    p.write_text(">a\n>b\nACGT\n>c\n")
    q = capi.Queries.from_file(str(p))
    assert q.labels == ["b", "c"] and list(q.arrays()[0]) == [0, 4, 4]
    assert capi.Queries.from_fasta(">a\n>b\nACGT\n>c\n").labels == ["b", "c"]


def test_bench_strong_scaling_slices_cover_the_job_once():
    """bench.py's partition of the default workload: every query of the job belongs to exactly one rank, at every N."""
    import bench

    for name in ("c3", "c4"):
        for world in (1, 2, 3, 4, 8):
            q_total, per, scaling = bench.workload_queries(name, world)
            assert scaling == "strong" and q_total == synth.CONFIGS[name][1]
            seen = 0
            for rank in range(world):
                q0 = min(rank * per, q_total)
                q1 = min(q0 + per, q_total)
                assert q0 == seen
                seen = q1
            assert seen == q_total
    q_total, per, scaling = bench.workload_queries("c2", 4)
    assert scaling == "weak" and per == synth.CONFIGS["c2"][1] and q_total == 4 * per
    assert bench.workload_queries("c5", 8, 131072) == (131072, 131072, "strong")  # sharded references: every rank sees every query


def test_bench_dump_outputs_bounded_and_reproducible(tmp_path):
    """bench.py --dump-outputs: float32 / float64 arrays only, at most the byte budget, the same files for the same results, every query
    while it all fits, and each dumped line the line of the query it is listed under."""
    import bench

    rng = np.random.default_rng(5)
    nq, ML = 3000, 6
    per_q = rng.integers(0, 9, nq)
    rb = np.concatenate([[0], np.cumsum(per_q)]).astype(np.uint32)
    n = int(rb[-1])
    lev = rng.integers(1, ML + 1, n).astype(np.uint8)
    out = capi.ClassifyOutput(rng.integers(0, 700, nq).astype(np.uint16), rb, rng.random(nq), rng.integers(0, 2**32 - 1, n, dtype=np.uint32),
                              lev, rng.random((n, ML)), rng.random(n))

    def load(d):
        return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}

    bench.dump_outputs(out, str(tmp_path / "all"))
    a = load(tmp_path / "all")
    assert set(a) == {"query", "n_kmers", "global_signal", "n_results", "first_ref", "n_levels", "confidence", "local_signal"}
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert np.array_equal(a["query"], np.arange(nq)) and np.array_equal(a["first_ref"], out.first_ref.astype(np.float64))
    assert np.array_equal(a["n_results"], per_q) and np.array_equal(a["n_kmers"], out.n_kmers)
    lv = np.arange(ML)[None, :] < lev[:, None]
    assert np.array_equal(a["confidence"][lv], out.confidence[lv]) and not a["confidence"][~lv].any()

    budget = 100_000
    for d in ("s1", "s2"):
        bench.dump_outputs(out, str(tmp_path / d), budget, first_query=10_000)
    s1, s2 = load(tmp_path / "s1"), load(tmp_path / "s2")
    assert all(np.array_equal(s1[k], s2[k]) for k in s1)
    assert 0 < len(s1["query"]) < nq and sum(v.nbytes for v in s1.values()) <= budget
    q = s1["query"].astype(np.int64) - 10_000
    assert np.all(np.diff(q) > 0) and np.array_equal(s1["n_results"], per_q[q])
    rows = np.concatenate([np.arange(rb[i], rb[i + 1]) for i in q])
    assert np.array_equal(s1["first_ref"], out.first_ref[rows]) and np.array_equal(s1["local_signal"], out.local_signal[rows])


def test_chunk_plan_covers_every_query_once():
    """rxh_plan_chunks (the driver's par_chunks, raxtax.rs:35-39): consecutive, non-empty chunks that cover [0, n) exactly; an explicit
    chunk size is kept as given; the library's own choice starts and ends every context's share of the job with small chunks."""
    for nq in (0, 1, 7, 999, 1024, 1025, 4096, 10_000, 25_000, 99_999, 200_000, 1_000_000):
        for n_ctx in (1, 2, 8):
            for cs in (0, 1, 64, 1000, 32768):
                b = capi.plan_chunks(nq, n_ctx, cs)
                assert b[0] == 0 and b[-1] == nq
                sizes = [b[i + 1] - b[i] for i in range(len(b) - 1)]
                assert all(x > 0 for x in sizes) and sum(sizes) == nq
                if cs:
                    assert all(x == cs for x in sizes[:-1]) and (not sizes or sizes[-1] <= cs)
                elif sizes:
                    assert max(sizes) <= 32768 * 3 // 2
    sizes = np.diff(capi.plan_chunks(200_000, 1, 0))
    assert sizes[0] < sizes[len(sizes) // 2] and sizes[-1] < sizes[len(sizes) // 2] and sizes[0] >= 1024
    sizes8 = np.diff(capi.plan_chunks(200_000, 8, 0))
    assert len(set(sizes8[:8])) == 1 and len(set(sizes8[-8:])) == 1  # one small first and last chunk per context


def test_host_tree_matches_oracle_on_random_degenerate_lineages(oracle):
    """Tree::new (tree.rs:47-140) on lineages drawn from a tiny label alphabet: repeated labels along a lineage, lineages that are
    prefixes of others (variable depth), empty levels, many identical lineages -- the cases in which the host's shared-prefix walk could
    part from the reference's "compare with the last child only" rule."""
    rng = np.random.default_rng(123)
    labels = ["a", "b", "ab", "", "a,", "c"]
    for case in range(60):
        n = int(rng.integers(1, 70))
        lineages = []
        for _ in range(n):
            depth = int(rng.integers(1, 6))
            lin = ",".join(labels[int(rng.integers(0, 4 if case % 2 else 3))].rstrip(",") for _ in range(depth))
            lineages.append(lin)
            if rng.random() < 0.3:
                lineages.append(lin)  # the same lineage again (several Sequence leaves under one taxon)
        seqs = [synth.BASE_CODES[rng.integers(0, 4, int(rng.integers(8, 24)))] for _ in lineages]
        off, codes = oracle.pack_sequences(seqs)
        _compare_tree(oracle.Tree.new(lineages, seqs), capi.Tree.new(lineages, off, codes))


def test_tree_build_pairwise_equals_level_walk(oracle):
    """The node tree built from consecutive lineage pairs (parallel string work + an integer pass, the default) is the tree the
    level-by-level walk of tree.rs:56-126 builds (RXH_TREE_WALK=1), on degenerate random lineages and on a synthetic set."""
    rng = np.random.default_rng(321)
    labels = ["a", "b", "ab", "", "c", "a!"]
    cases = []
    for case in range(80):
        lineages = []
        for _ in range(int(rng.integers(1, 120))):
            lin = ",".join(labels[int(rng.integers(0, 3 + case % 4))] for _ in range(int(rng.integers(1, 6))))
            lineages += [lin] * int(rng.integers(1, 4))
        rng.shuffle(lineages)
        cases.append(lineages)
    ds = synth.generate("small", n_queries=1, measure=False)
    cases.append(list(ds.ref_lineages))
    for lineages in cases:
        seqs = [synth.BASE_CODES[rng.integers(0, 4, 12)] for _ in lineages]
        off, codes = oracle.pack_sequences(seqs)
        a = capi.Tree.new(lineages, off, codes).index_arrays()
        os.environ["RXH_TREE_WALK"] = "1"
        try:
            b = capi.Tree.new(lineages, off, codes).index_arrays()
        finally:
            del os.environ["RXH_TREE_WALK"]
        assert a.keys() == b.keys()
        for k in a:
            assert np.array_equal(a[k], b[k]), k
