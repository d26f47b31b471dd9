"""Generates tests/golden/diptera_sample.fasta: the first 400 records of the reference repository's example data
(example/diptera_queries.fasta, the only example file shipped; SURVEY.md 8(c) uses it as its own database).
Usage: make_diptera_sample.py <reference checkout>/example/diptera_queries.fasta; the tests read the committed sample only."""
import os
import sys

DST = os.path.join(os.path.dirname(os.path.abspath(__file__)), "diptera_sample.fasta")
N = 400

if __name__ == "__main__":
    out, n = [], 0
    for line in open(sys.argv[1]):
        if line.startswith(">"):
            n += 1
            if n > N:
                break
        out.append(line)
    open(DST, "w").write("".join(out))
    print(DST, n - 1 if n > N else n, "records")
