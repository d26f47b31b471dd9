"""Generates tests/golden/diptera_queries.fasta.gz: the reference repository's whole example file (example/diptera_queries.fasta,
7 868 records), gzip-compressed -- BASELINE config 1 in the form SURVEY.md 8(c) prescribes (the file used as its own database, default
and --skip-exact-matches).  Usage: make_diptera_full.py <reference checkout>/example/diptera_queries.fasta; the tests read the
committed copy only."""
import gzip
import os
import sys

DST = os.path.join(os.path.dirname(os.path.abspath(__file__)), "diptera_queries.fasta.gz")

if __name__ == "__main__":
    data = open(sys.argv[1], "rb").read()
    with gzip.GzipFile(DST, "wb", compresslevel=9, mtime=0) as f:
        f.write(data)
    print(DST, len(data), "->", os.path.getsize(DST), "bytes,", data.count(b">"), "records")
