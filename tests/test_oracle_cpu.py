"""CPU suite (-m "not gpu"): the oracle against the reference's golden matrices, host logic, ABI surface."""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import GOLDEN, REF_TEST_DIR, ROOT, golden_dict, same_entries, triplet_dict, to_oracle_batch


def test_oracle_reproduces_goldens_from_committed_fixtures(oracle, goldens, golden_batches):
    """All 12 golden comparisons of main.rs:1207-1466, from the staged fixtures in tests/golden."""
    for case in goldens["cases"]:
        batch = golden_batches[case["batch"]]
        bcs = oracle.Barcodes([k.encode() for k in goldens["barcodes"][case["barcodes"]]])
        res = oracle.run_batch(batch, bcs, oracle.MODES[case["scoring_method"]], case["umi"])
        g = goldens["matrices"][case["out"]]
        assert (batch.n_rows, len(bcs)) == (g["n_rows"], g["n_cols"]), case["name"]
        assert same_entries(triplet_dict(res.row, res.col, res.val), golden_dict(g)), case["name"]
        if case["ref"]:
            g2 = goldens["matrices"][case["ref"]]
            assert same_entries(triplet_dict(res.row, res.col, res.val2), golden_dict(g2)), case["name"]


@pytest.mark.skipif(not os.path.isdir(REF_TEST_DIR), reason="tests/golden/ref_inputs missing")
def test_oracle_reproduces_goldens_from_reference_files(oracle):
    from oracle import check_goldens
    assert check_goldens.main(REF_TEST_DIR) == 0


@pytest.mark.skipif(not os.path.isdir(REF_TEST_DIR), reason="tests/golden/ref_inputs missing")
def test_committed_fixtures_are_current(oracle, golden_batches):
    b = oracle.stage_from_files(f"{REF_TEST_DIR}/test_dna.vcf", f"{REF_TEST_DIR}/test_dna.bam", f"{REF_TEST_DIR}/test_dna.fa")
    g = golden_batches["dna_batch.npz"]
    for f in oracle.Batch.FIELDS:
        assert np.array_equal(getattr(b, f), getattr(g, f)), f


def test_sw_known_answers(oracle):
    sw = oracle.sw_full
    assert sw(b"ACGTACGTAC", b"ACGTACGTAC") == 10
    assert sw(b"ACGTACGTAC", b"TTTTACGTACGTACTTTT") == 10
    assert sw(b"AAAAAAAAAA", b"CCCCCCCCCC") == 0
    assert sw(b"", b"ACGT") == 0
    # one mismatch in the middle of 20 matches: 10 + 10 - 5 = 15 beats either side alone (10)
    assert sw(b"ACGTACGTAC" + b"G" + b"TTGACCATGA", b"ACGTACGTAC" + b"C" + b"TTGACCATGA") == 15
    # gap of length 2 costs 5 + 2 = 7
    assert sw(b"ACGTACGTACGGATCCATTG" + b"TTGACCATGATTGACAGGTA", b"ACGTACGTACGGATCCATTG" + b"CC" + b"TTGACCATGATTGACAGGTA") == 33
    # byte equality: lower case never matches upper case (main.rs:898, A.5)
    assert sw(b"ACGTACGT", b"acgtacgt") == 0


def test_evaluate_scores_table(oracle):
    ev = oracle.lib().vtxo_evaluate_scores
    assert ev(24, 24) == 0 and ev(25, 24) == 1 and ev(24, 25) == 2 and ev(25, 25) == -1
    assert ev(100, 94) == 1 and ev(94, 100) == 2 and ev(0, 0) == 0


def test_useful_alignment_cigar_rules(oracle):
    ua = oracle.lib().vtxo_useful_alignment
    def cig(*ops):
        code = {"M": 0, "I": 1, "D": 2, "N": 3, "S": 4, "H": 5, "P": 6, "=": 7, "X": 8}
        a = np.array([(n << 4) | code[o] for n, o in ops], np.uint32)
        return a, a.ctypes.data, len(a)
    a, p, n = cig((50, "M"))
    assert ua(100, p, n, 120, 121) == 1 and ua(100, p, n, 149, 150) == 1
    assert ua(100, p, n, 150, 151) == 0 and ua(100, p, n, 98, 99) == 0 and ua(100, p, n, 99, 100) == 1   # inclusive end (main.rs:794)
    a, p, n = cig((10, "M"), (100, "N"), (10, "M"))                           # spliced-over locus is not covered
    assert ua(100, p, n, 150, 151) == 0 and ua(100, p, n, 210, 211) == 1
    a, p, n = cig((10, "M"), (5, "D"), (10, "M"))                             # deletions count
    assert ua(100, p, n, 112, 113) == 1
    a, p, n = cig((5, "S"), (10, "M"))                                        # soft clips do not
    assert ua(100, p, n, 95, 98) == 0 and ua(100, p, n, 100, 101) == 1
    a, p, n = cig((5, "D"), (10, "M"))                                        # leading D -> error -> skipped
    assert ua(100, p, n, 100, 101) == 0


def test_band_model_equals_full_on_fixture_pairs(oracle, golden_batches, goldens):
    """SURVEY.md Appendix C: under the golden-consistent band model no fixture pair loses score."""
    b = golden_batches["dna_batch.npz"]
    bcs = oracle.Barcodes([k.encode() for k in goldens["barcodes"]["dna_barcodes.tsv"]])
    full = oracle.run_batch(b, bcs, oracle.MODE_COVERAGE, False)
    band = oracle.run_batch(b, bcs, oracle.MODE_COVERAGE, False, band_model=True)
    assert np.array_equal(full.val, band.val) and np.array_equal(full.val2, band.val2)


def test_oracle_threads_do_not_change_results(oracle):
    import vartrix_b200 as vb
    sb, bcs, info = vb.synth.make_shard(64, 40, depth=20, seed=5)
    ob = to_oracle_batch(oracle, sb); obc = oracle.Barcodes(bcs.keys)
    a = oracle.run_batch(ob, obc, oracle.MODE_ALT_FRAC, False, n_threads=1)
    b = oracle.run_batch(ob, obc, oracle.MODE_ALT_FRAC, False, n_threads=5)      # 64 / 5 -> 6 chunks (main.rs:250-254)
    assert np.array_equal(a.row, b.row) and np.array_equal(a.col, b.col) and np.array_equal(a.val, b.val, equal_nan=True)
    assert a.metrics["num_scored"] == info["n_pairs"]


def test_mtx_text_matches_sprs_layout(oracle):
    import vartrix_b200 as vb
    for mod in (oracle, vb.mtx):
        txt = mod.mtx_text(4, 20, [0, 1], [19, 14], [0.0, 1.0])
        assert txt == "%%MatrixMarket matrix coordinate real general\n% written by sprs\n4 20 2\n1 20 0\n2 15 1\n"
        f = mod.fmt_f64
        assert f(0.5) == "0.5" and f(1 / 3) == "0.3333333333333333" and f(float("nan")) == "NaN" and f(7.0) == "7"
        assert f(1e-6) == "0.000001" and f(2 / 3) == "0.6666666666666666"


def test_header_symbols_are_exported():
    """The C-ABI library loads on a CPU-only box and exports every function include/vartrix_b200.h declares."""
    from vartrix_b200 import _capi
    hdr = open(os.path.join(ROOT, "include", "vartrix_b200.h")).read()
    declared = set(re.findall(r"\b(vtx_[a-z0-9_]+)\s*\(", hdr))
    declared = {d for d in declared if not d.startswith("vtx_k_")}      # kernel names cited in comments
    assert declared == set(_capi.SYMBOLS), declared ^ set(_capi.SYMBOLS)
    lib = ctypes.CDLL(_capi.LIB_PATH)
    for s in _capi.SYMBOLS:
        assert hasattr(lib, s), s
    assert lib.vtx_abi_version() == 2


def test_header_is_plain_c(tmp_path):
    """The boundary is a C ABI: the header must compile as C99 (no C++-isms, no torch / CUDA types) and link against
    the library from a C translation unit."""
    import subprocess
    from vartrix_b200 import _capi
    src = tmp_path / "abi.c"
    src.write_text('#include "vartrix_b200.h"\n'
                   'int main(void) { vtx_config c; vtx_batch b; vtx_batch2 b2; vtx_result r; vtx_timing t; (void)c; (void)b; (void)b2; (void)r; (void)t;\n'
                   '  return vtx_abi_version() == 2 && vtx_pack_cb((const unsigned char*)"ACGT-1", 6) == 111105ull && vtx_pack_umi((const unsigned char*)"ACGT", 4) != VTX_NO_UMI ? 0 : 1; }\n')
    exe = tmp_path / "abi"
    libdir = os.path.dirname(_capi.LIB_PATH)
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                    "-L", libdir, "-lvartrix_b200", f"-Wl,-rpath,{libdir}"], check=True)
    assert subprocess.run([str(exe)]).returncode == 0


def test_engine_fails_loudly_without_gpu():
    import vartrix_b200 as vb
    from conftest import HAS_GPU
    if HAS_GPU:
        pytest.skip("GPU present")
    with pytest.raises(vb.VtxError, match="no CUDA device|CPU fallback|failed"):
        vb.Engine("coverage")


def test_pack_umi_is_injective_and_matches_synth():
    import vartrix_b200 as vb
    assert vb.pack_umi(b"ACGTACGTAC") == (int("".join("{:03b}".format("ACGTN".index(c)) for c in "ACGTACGTAC"), 2) << 5) | 10
    assert vb.pack_umi(b"ACGT") != vb.pack_umi(b"AACGT") != vb.pack_umi(b"ACGTA")
    assert vb.pack_umi(b"ACGU") == vb.NO_UMI if hasattr(vb, "NO_UMI") else True
    assert vb.pack_umi(b"A" * 19) == 0xFFFFFFFFFFFFFFFF and vb.pack_umi(b"T" * 18) < 2**59


def test_synth_shapes_and_shard_invariance(oracle):
    import vartrix_b200 as vb
    sb, bcs, info = vb.synth.make_shard(30, 25, depth=12, seed=9, kind="indel", umi=True)
    assert sb.n_cand == 30 * 12 and info["max_hap_len"] <= 231 and (sb.ref_off % 16 == 0).all() and (sb.read_off % 16 == 0).all()
    assert (np.abs(sb.ref_len.astype(int) - sb.alt_len.astype(int)) >= 1).all()      # every locus is an indel
    obc = oracle.Barcodes(bcs.keys)
    whole = oracle.run_batch(to_oracle_batch(oracle, sb), obc, oracle.MODE_COVERAGE, True)
    parts = [oracle.run_batch(to_oracle_batch(oracle, sb.shard(lo, hi)), obc, oracle.MODE_COVERAGE, True)
             for lo, hi in vb.shard_bounds(sb.cand_start, 3)]
    for f in ("row", "col", "val", "val2"):
        assert np.array_equal(np.concatenate([getattr(p, f) for p in parts]), getattr(whole, f)), f
    assert vb.shard_bounds(sb.cand_start, 3)[0][0] == 0 and vb.shard_bounds(sb.cand_start, 3)[-1][1] == 30


def test_shard_schedules_cover_every_locus_once():
    import vartrix_b200 as vb
    rng = np.random.default_rng(4)
    cs = np.concatenate([[0], np.cumsum(rng.integers(0, 90, size=5000))]).astype(np.uint64)
    for kw in (dict(n_shards=1), dict(n_shards=7), dict(n_shards=8, first_frac=0.02), dict(n_shards=6, first_frac=0.01, growth=1.4),
               dict(n_shards=6, first_frac=0.01, growth=1.1), dict(n_shards=3, first_frac=0.5, growth=1.4)):
        b = vb.shard_bounds(cs, **kw)
        assert b[0][0] == 0 and b[-1][1] == 5000 and all(b[i][1] == b[i + 1][0] for i in range(len(b) - 1)), kw
        assert all(hi >= lo for lo, hi in b), kw
    geo = vb.shard_bounds(cs, 6, first_frac=0.01, growth=1.4)
    sizes = [int(cs[hi] - cs[lo]) for lo, hi in geo]
    total = int(cs[-1])
    assert sizes[0] <= 0.012 * total + 90 and max(sizes) <= total / 6 + 180          # primer, then capped at 1/6 of the step
    assert all(sizes[i + 1] <= 1.4 * sizes[i] + 180 for i in range(len(sizes) - 2))   # each copy hides behind the shard before it


def test_band_model_equals_full_on_synthetic_shards(oracle):
    """DESIGN.md 2: on the synthetic workloads (random context, SNVs and <= 30 bp indels) the best-effort model of
    rust-bio's k=6 / w=20 band never clips the optimal path, so full-matrix scores are the banded scores."""
    import vartrix_b200 as vb
    for kind in ("snv", "indel"):
        sb, bcs, _ = vb.synth.make_shard(24, 30, depth=20, seed=31, kind=kind)
        ob = to_oracle_batch(oracle, sb); obc = oracle.Barcodes(bcs.keys)
        full = oracle.run_batch(ob, obc, oracle.MODE_COVERAGE, False, n_threads=4)
        band = oracle.run_batch(ob, obc, oracle.MODE_COVERAGE, False, n_threads=4, band_model=True)
        assert np.array_equal(full.val, band.val) and np.array_equal(full.val2, band.val2) and np.array_equal(full.unk_cnt, band.unk_cnt), kind


def test_bench_arguments_and_shard_growth_policy():
    """bench.py parses on a CPU-only box, and its shard-growth policy stays inside [1.1, cap]."""
    import importlib.util
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True)
    assert r.returncode == 0 and "--impl" in r.stdout and "--growth" in r.stdout
    spec = importlib.util.spec_from_file_location("vtx_bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec); spec.loader.exec_module(mod)
    assert mod.pick_growth(16.6, 35.3, 1.4) == 1.4            # one GPU: copies are twice as fast as the kernels
    assert 1.15 < mod.pick_growth(27.0, 36.6, 1.4) < 1.3      # eight ranks sharing the host's PCIe paths
    assert mod.pick_growth(80.0, 36.0, 1.4) == 1.1 and mod.pick_growth(0.0, 1.0, 1.4) == 1.4
    assert mod.parse_args(["--steps", "7"]).steps == 7
    with pytest.raises(SystemExit):
        mod.parse_args(["--steps", "0"])


def test_bench_dump_outputs_is_a_fixed_capped_sample(tmp_path):
    """bench.py --dump-outputs: float64 arrays of whole triplets at the same seeded positions every run, 64 MB at most."""
    import importlib.util
    import vartrix_b200 as vb
    spec = importlib.util.spec_from_file_location("vtx_bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec); spec.loader.exec_module(mod)
    rng = np.random.default_rng(1)
    n = mod.DUMP_MAX_ENTRIES + 12345
    row = np.sort(rng.integers(0, 1 << 31, n)).astype(np.uint32)
    col = rng.integers(0, 1 << 31, n).astype(np.uint32)
    none = np.zeros(0, np.uint32)
    res = vb.Triplets(row, col, none, none, none, row * 0.5 + col, -1.0 * col, dict(num_scored=7, num_not_cell_bc=8, num_non_umi=9))
    for d in ("a", "b"):
        mod.dump_outputs(str(tmp_path / d), res, True)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["col.npy", "metrics.npy", "row.npy", "val.npy", "val2.npy"]
    got = {}
    for nm in names:
        a, b = np.load(tmp_path / "a" / nm), np.load(tmp_path / "b" / nm)
        assert a.dtype == np.float64 and np.array_equal(a, b), nm
        got[nm[:-4]] = a
    assert sum(os.path.getsize(tmp_path / "a" / nm) for nm in names) <= 64 << 20
    assert len(got["row"]) == mod.DUMP_MAX_ENTRIES and (np.diff(got["row"]) >= 0).all()        # sampled in triplet order
    assert np.array_equal(got["val"], got["row"] * 0.5 + got["col"]) and np.array_equal(got["val2"], -got["col"])
    assert np.array_equal(got["metrics"], [n, 7, 8, 9])
    small = vb.Triplets(row[:10], col[:10], none, none, none, res.val[:10], none.astype(np.float64), res.metrics)
    mod.dump_outputs(str(tmp_path / "small"), small, False)
    assert sorted(os.listdir(tmp_path / "small")) == ["col.npy", "metrics.npy", "row.npy", "val.npy"]
    assert np.array_equal(np.load(tmp_path / "small" / "row.npy"), row[:10])
