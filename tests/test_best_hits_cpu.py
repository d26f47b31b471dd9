"""--best-hits without a GPU: the declared ABI of the feature and the CLI's handling of the flag -- usage errors before any input is
read, the checkpoint key and the resume rule, --help."""
import json
import os
import re
import subprocess

from raxtax_b200 import _build, capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FASTA = os.path.join(ROOT, "tests", "golden", "diptera_sample.fasta")


def _cli(*args):
    return subprocess.run([_build.CLI_BIN, *map(str, args)], capture_output=True, text=True)


def test_best_hits_abi_is_declared():
    h = open(os.path.join(ROOT, "include", "raxtax_b200.h")).read()
    assert re.search(r"RTX_OPT_BEST_HITS = 12\b", h)
    assert capi.RTX_OPT_BEST_HITS == 12
    assert "int rtx_batch_best_hits(rtx_ctx* ctx, uint32_t* n_hits" in h
    assert "rtx_batch_best_hits" in capi.DEVICE_SYMBOLS
    hh = open(os.path.join(ROOT, "include", "raxtax_host.h")).read()
    assert "typedef int (*rxh_hits_sender)(void* user, const char* query_label, const char* hit_lines);" in hh
    assert "int rxh_raxtax_best_hits(" in hh and "rxh_raxtax_best_hits" in capi.HOST_SYMBOLS
    assert hasattr(capi.device_lib(), "rtx_batch_best_hits") and hasattr(capi.host_lib(), "rxh_raxtax_best_hits")


def test_cli_rejects_bad_best_hits_values(tmp_path):
    for v in ("0", "65", "-1", "ten", "", "5x", "1e1", "100"):
        r = _cli("-d", FASTA, "-i", FASTA, "-o", tmp_path / "o", "--best-hits", v)
        assert r.returncode == 64, (v, r.stderr)
        assert "--best-hits" in r.stderr, v
        assert not (tmp_path / "o").exists(), v  # nothing was read or written
    r = _cli("-d", FASTA, "-i", FASTA, "-o", tmp_path / "o", "--best-hits")
    assert r.returncode == 64 and "--best-hits" in r.stderr and not (tmp_path / "o").exists()


def test_cli_rejects_best_hits_with_sharded_references(tmp_path):
    for gpus in (["--gpus", "2"], []):
        r = _cli("-d", FASTA, "-i", FASTA, "-o", tmp_path / "o", *gpus, "--shard-references", "--best-hits", "5")
        assert r.returncode == 64, r.stderr
        assert "--best-hits" in r.stderr and "--shard-references" in r.stderr
        assert not (tmp_path / "o").exists()


def test_cli_checkpoint_records_best_hits_only_when_set(tmp_path):
    r = _cli("--only-db", "-d", FASTA, "-o", tmp_path / "plain")
    assert r.returncode == 0, r.stderr
    assert "best_hits" not in json.loads((tmp_path / "plain" / "raxtax.json").read_text())
    r = _cli("--only-db", "--best-hits", "7", "-d", FASTA, "-o", tmp_path / "hits")
    assert r.returncode == 0, r.stderr
    ck = json.loads((tmp_path / "hits" / "raxtax.json").read_text())
    assert ck["best_hits"] == 7 and ck["tsv"] is False and "strand" not in ck
    # the same run again resumes from its checkpoint; a run with another value -- or without the flag -- finds the checkpoint invalid,
    # as one with another --tsv setting does, and starts over from the FASTA, whose database already exists
    r = _cli("--only-db", "--best-hits", "7", "-d", FASTA, "-o", tmp_path / "hits")
    assert r.returncode == 0, r.stderr
    for other in (["--best-hits", "8"], [], ["--best-hits", "7", "--tsv"]):
        r = _cli("--only-db", *other, "-d", FASTA, "-o", tmp_path / "hits")
        assert r.returncode != 0 and "already exists" in r.stderr, (other, r.stderr)
    # and a checkpoint written without the flag is not resumed with it
    r = _cli("--only-db", "--best-hits", "1", "-d", FASTA, "-o", tmp_path / "plain")
    assert r.returncode != 0 and "already exists" in r.stderr, r.stderr


def test_cli_help_lists_best_hits():
    r = _cli("--help")
    assert r.returncode == 0 and "--best-hits <N>" in r.stderr
