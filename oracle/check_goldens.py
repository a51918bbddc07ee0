"""CPU ORACLE (test infrastructure): pin the oracle against the reference's own golden matrices.

Runs the seven regression cases of /root/reference/src/main.rs:1207-1466 through
oracle.pipeline (Python decode + C oracle) and compares every output with the committed
golden `.mtx` as a (row, col) -> value set, exactly like the reference's
`assert_eq!(seen.to_csr(), expected.to_csr())` (main.rs:1230-1232).

Usage:  python -m oracle.check_goldens [reference_test_dir]      (default tests/golden/ref_inputs)
"""
import math
import os
import sys

from . import pipeline as P

REF_TEST_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "ref_inputs")

CASES = [  # (name, main.rs lines, files prefix, barcodes, mode, umi, golden out, golden ref)
    ("test_consensus_matrix", "1207-1233", "test", "barcodes.tsv", "consensus", False, "test_consensus.mtx", None),
    ("test_frac_matrix", "1235-1263", "test", "barcodes.tsv", "alt_frac", False, "test_frac.mtx", None),
    ("test_coverage_matrices", "1265-1300", "test", "barcodes.tsv", "coverage", False, "test_coverage.mtx", "test_coverage_ref.mtx"),
    ("test_coverage_matrices_umi", "1302-1339", "test", "barcodes.tsv", "coverage", True, "test_coverage_umi.mtx", "test_coverage_ref_umi.mtx"),
    ("test_coverage_matrices_umi_gzipped_bcs", "1341-1390", "test", "barcodes.tsv.gz", "coverage", True, "test_coverage_umi.mtx", "test_coverage_ref_umi.mtx"),
    ("test_coverage_matrices_umi_dna", "1392-1429", "test_dna", "dna_barcodes.tsv", "coverage", True, "test_dna_umi.mtx", "test_dna_ref_umi.mtx"),
    ("test_coverage_matrices_dna", "1431-1466", "test_dna", "dna_barcodes.tsv", "coverage", False, "test_dna.mtx", "test_dna_ref.mtx"),
]


def triplets(res, which="val"):
    d = {}
    for r, c, v in zip(res.row, res.col, getattr(res, which)):
        d[(int(r), int(c))] = d.get((int(r), int(c)), 0.0) + float(v)
    return d


def same(a, b):
    if a.keys() != b.keys():
        return False
    return all((math.isnan(a[k]) and math.isnan(b[k])) or a[k] == b[k] for k in a)


def main(test_dir=REF_TEST_DIR):
    ok = True
    for name, lines, pre, bcs, mode, umi, g_out, g_ref in CASES:
        nr, nc, res, batch, _ = P.run_files(f"{test_dir}/{pre}.vcf", f"{test_dir}/{pre}.bam", f"{test_dir}/{pre}.fa",
                                            f"{test_dir}/{bcs}", mode, umi)
        gr, gc, gent = P.read_mtx(f"{test_dir}/{g_out}")
        good = (nr, nc) == (gr, gc) and same(triplets(res), gent)
        if g_ref:
            gr2, gc2, gent2 = P.read_mtx(f"{test_dir}/{g_ref}")
            good = good and (nr, nc) == (gr2, gc2) and same(triplets(res, "val2"), gent2)
        print(f"{'PASS' if good else 'FAIL'}  {name} (main.rs:{lines})  fetched={batch.host_metrics['num_reads']} "
              f"cand={batch.n_cand} scored={res.metrics['num_scored']} nnz={len(res.row)}")
        ok &= good
    print("ALL 12 GOLDENS REPRODUCED" if ok else "GOLDEN MISMATCH")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main(*sys.argv[1:]))
