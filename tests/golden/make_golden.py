"""Regenerates tests/golden/*.npz|json from the reference's own fixtures (by default the verbatim copy of the
reference's test/ directory in tests/golden/ref_inputs).

  python tests/golden/make_golden.py [reference_test_dir]

Outputs
  rna_batch.npz / dna_batch.npz : the staged candidates of test/test.{vcf,bam,fa} and test/test_dna.*
                                  (oracle.pipeline.stage_from_files = main.rs up to the CB lookup)
  goldens.json                  : the 12 golden matrices of the reference (test/*.mtx) as triplets,
                                  the barcode lists, and the driving argv of each regression test
                                  (main.rs:1207-1466)
"""
import json
import os
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))
from oracle import pipeline as P          # noqa: E402
from oracle.check_goldens import CASES    # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def main(test_dir=os.path.join(HERE, "ref_inputs")):
    for pre, out in (("test", "rna_batch.npz"), ("test_dna", "dna_batch.npz")):
        b = P.stage_from_files(f"{test_dir}/{pre}.vcf", f"{test_dir}/{pre}.bam", f"{test_dir}/{pre}.fa")
        b.save(os.path.join(HERE, out))
        print(out, "loci", b.n_loci, "reads", b.n_reads, "cand", b.n_cand, b.host_metrics)
    g = {"barcodes": {}, "cases": [], "matrices": {}}
    for name in ("barcodes.tsv", "barcodes.tsv.gz", "dna_barcodes.tsv"):
        g["barcodes"][name] = [k.decode() for k in P.load_barcodes(f"{test_dir}/{name}").keys]
    for name, lines, pre, bcs, mode, umi, g_out, g_ref in CASES:
        g["cases"].append(dict(name=name, main_rs=lines, batch=("rna_batch.npz" if pre == "test" else "dna_batch.npz"),
                               barcodes=bcs, scoring_method=mode, umi=umi, out=g_out, ref=g_ref))
        for m in (g_out, g_ref):
            if m and m not in g["matrices"]:
                nr, nc, ent = P.read_mtx(f"{test_dir}/{m}")
                g["matrices"][m] = dict(n_rows=nr, n_cols=nc,
                                        entries=sorted([r, c, v] for (r, c), v in ent.items()))
    for m in ("test_consensus.mtx", "test_frac.mtx"):
        assert m in g["matrices"]
    with open(os.path.join(HERE, "goldens.json"), "w") as fh:
        json.dump(g, fh, indent=0, separators=(",", ":"))
    print("goldens.json:", len(g["matrices"]), "matrices,", len(g["cases"]), "cases")


if __name__ == "__main__":
    main(*sys.argv[1:])
