"""--strand both without a GPU: the reverse-complement helpers, the 8-mer identity the device relies on (the k-mer set of rc(s) is
rc16 of the k-mer set of s, so n_kmers does not depend on the strand) and the declared ABI of the feature."""
import os
import re

import numpy as np

from raxtax_b200 import capi, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# IUPAC code -> code of its complement (parser.rs:11-34 bit assignment A1 C2 G4 T8)
COMPLEMENT_TABLE = {"A": "T", "C": "G", "G": "C", "T": "A", "R": "Y", "Y": "R", "S": "S", "W": "W", "K": "M", "M": "K", "B": "V",
                    "V": "B", "D": "H", "H": "D", "N": "N"}


def rc16(k):
    """Reverse complement of a 2-bit packed 8-mer (first base in bits 15..14)."""
    x = k ^ 0xFFFF
    return int("".join(f"{x:016b}"[i: i + 2] for i in range(14, -2, -2)), 2)


def test_complement_table_all_15_codes():
    char_to_code = {c: k for k, c in synth.CODE_TO_CHAR.items()}
    assert len(char_to_code) == 15
    for c, comp in COMPLEMENT_TABLE.items():
        assert synth.COMPLEMENT[char_to_code[c]] == char_to_code[comp], c
    assert synth.COMPLEMENT[0] == 0


def test_reverse_complement_is_an_involution():
    rng = np.random.default_rng(3)
    s = rng.integers(1, 16, 1001).astype(np.uint8)
    assert np.array_equal(synth.reverse_complement(synth.reverse_complement(s)), s)
    assert list(synth.reverse_complement(np.array([1, 1, 2, 4, 5], np.uint8))) == [10, 2, 4, 8, 8]  # AACGR -> YCGTT
    off = np.array([0, 5, 5, 12, 20], np.uint64)
    codes = rng.integers(1, 16, 20).astype(np.uint8)
    which = np.array([True, False, True, False])
    once = synth.reverse_complement_batch(off, codes, which)
    for i in range(4):
        a, b = int(off[i]), int(off[i + 1])
        exp = synth.reverse_complement(codes[a:b]) if which[i] else codes[a:b]
        assert np.array_equal(once[a:b], exp)
    assert np.array_equal(synth.reverse_complement_batch(off, once, which), codes)
    assert np.array_equal(synth.reverse_complement_batch(off, synth.reverse_complement_batch(off, codes), None), codes)


def test_kmers_of_reverse_complement_are_rc16_of_kmers():
    ds = synth.generate("tiny", measure=False)
    for i in range(0, ds.n_queries, 7):
        s = ds.query_seq(i)
        k = synth.kmers_of(s)
        krc = synth.kmers_of(synth.reverse_complement(s))
        assert len(k) == len(krc)
        assert np.array_equal(np.sort(np.array([rc16(int(x)) for x in k], np.uint16)), krc)
    assert rc16(0x0000) == 0xFFFF  # AAAAAAAA <-> TTTTTTTT
    assert rc16(0x1B1B) == 0x1B1B  # ACGTACGT is its own reverse complement


def test_both_strands_abi_is_declared():
    h = open(os.path.join(ROOT, "include", "raxtax_b200.h")).read()
    assert re.search(r"#define RTX_BOTH_STRANDS 4u", h)
    assert capi.RTX_BOTH_STRANDS == 4
    assert "int rtx_batch_strands(rtx_ctx* ctx, uint8_t* strand" in h
    assert "rtx_batch_strands" in capi.DEVICE_SYMBOLS


# ---- CLI: --strand <plus|both> (vsearch's spelling), checked before any input is read ---------------------------------------------
FASTA = os.path.join(ROOT, "tests", "golden", "diptera_sample.fasta")


def _cli(*args):
    import subprocess

    from raxtax_b200 import _build

    return subprocess.run([_build.CLI_BIN, *map(str, args)], capture_output=True, text=True)


def test_cli_rejects_bad_strand_value(tmp_path):
    r = _cli("-d", FASTA, "-i", FASTA, "-o", tmp_path / "o", "--strand", "minus")
    assert r.returncode == 64, r.stderr
    assert "--strand" in r.stderr and "plus, both" in r.stderr
    assert not (tmp_path / "o").exists()  # nothing was read or written
    r = _cli("-d", FASTA, "-i", FASTA, "-o", tmp_path / "o", "--strand")
    assert r.returncode == 64 and not (tmp_path / "o").exists()


def test_cli_rejects_both_strands_with_sharded_references(tmp_path):
    r = _cli("-d", FASTA, "-i", FASTA, "-o", tmp_path / "o", "--gpus", 2, "--shard-references", "--strand", "both")
    assert r.returncode == 64, r.stderr
    assert "--shard-references" in r.stderr
    assert not (tmp_path / "o").exists()


def test_cli_checkpoint_records_strand_only_in_both_mode(tmp_path):
    import json

    r = _cli("--only-db", "-d", FASTA, "-o", tmp_path / "plain")
    assert r.returncode == 0, r.stderr
    assert "strand" not in json.loads((tmp_path / "plain" / "raxtax.json").read_text())
    r = _cli("--only-db", "--strand", "plus", "-d", FASTA, "-o", tmp_path / "plus")
    assert r.returncode == 0, r.stderr
    assert "strand" not in json.loads((tmp_path / "plus" / "raxtax.json").read_text())
    r = _cli("--only-db", "--strand", "both", "-d", FASTA, "-o", tmp_path / "both")
    assert r.returncode == 0, r.stderr
    ck = json.loads((tmp_path / "both" / "raxtax.json").read_text())
    assert ck["strand"] == "both" and ck["tsv"] is False
    # the same run again resumes from its checkpoint (the database is read back from the .bin it points to); a run with the other
    # strand setting finds the checkpoint invalid -- as one with another --tsv setting does -- and starts over from the FASTA, whose
    # database already exists
    r = _cli("--only-db", "--strand", "both", "-d", FASTA, "-o", tmp_path / "both")
    assert r.returncode == 0, r.stderr
    for other in (["--strand", "plus"], ["--strand", "both", "--tsv"]):
        r = _cli("--only-db", *other, "-d", FASTA, "-o", tmp_path / "both")
        assert r.returncode != 0 and "already exists" in r.stderr, (other, r.stderr)


def test_cli_help_lists_strand():
    r = _cli("--help")
    assert r.returncode == 0 and "--strand <STRAND>" in r.stderr
